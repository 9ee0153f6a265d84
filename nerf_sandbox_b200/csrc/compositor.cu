// K3 -- alpha compositor, forward and backward, one warp per ray.
// Restates volume_render_rays (utils/render_utils.py:108-167) and, in the RAW variants, the head
// activations of nerf_forward_pass (:236-246) so that raw MLP logits are consumed directly.
// The exclusive cumprod transmittance is a multiplicative warp scan carried across 32-sample chunks;
// rgb/depth/acc reductions ride the same pass.  The backward recomputes T (never reads it from HBM),
// stages alpha/T per warp in shared memory and walks the ray in reverse with a suffix-sum scan.
#include "nsb_common.cuh"

namespace nsb {

constexpr int kCompWarps = 4;

struct Sample { float r, g, b, sigma; };

// RAW=false: rgb[B,N,3], sigma[B,N].  RAW=true: raw[B*N,4] logits (+ optional noise).
template <bool RAW>
__device__ __forceinline__ Sample load_sample(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma,
                                              const float* __restrict__ noise, float noise_std, bool add_noise,
                                              uint64_t seed, uint64_t offset, int64_t q, float* pre_out,
                                              const float* pre_in = nullptr, bool softplus = false, int64_t idx0 = 0) {
    Sample s;
    if (RAW) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(rgb_or_raw) + q);
        s.r = 1.0f / (1.0f + expf(-v.x));                     // :236 sigmoid
        s.g = 1.0f / (1.0f + expf(-v.y));
        s.b = 1.0f / (1.0f + expf(-v.z));
        float pre = v.w;
        if (pre_in) pre = *pre_in;                            // reverse pass: noisy pre-activation kept from pass 1
        else if (add_noise) pre += (noise ? noise[q] : hash_normal(seed, offset, (uint64_t)(q + idx0))) * noise_std;   // :239-241
        if (pre_out) *pre_out = pre;
        // :243-246 relu, or F.softplus (beta = 1, threshold = 20: identity above it)
        s.sigma = softplus ? (pre > 20.0f ? pre : log1pf(expf(pre))) : fmaxf(pre, 0.0f);
    } else {
        s.r = rgb_or_raw[q * 3 + 0]; s.g = rgb_or_raw[q * 3 + 1]; s.b = rgb_or_raw[q * 3 + 2];
        s.sigma = sigma[q];
    }
    return s;
}

__device__ __forceinline__ float delta_at(const float* __restrict__ zrow, int i, int N, bool inf_last, float rn,
                                          bool has_rn) {
    float d = (i == N - 1) ? (inf_last ? 1e10f : 0.0f) : (zrow[i + 1] - zrow[i]);   // :131-136
    if (has_rn) d *= rn;                                                               // :139-141
    return d;
}

// inclusive multiplicative scan across the warp
__device__ __forceinline__ float warp_scan_mul(float v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v *= t;
    }
    return v;
}

__device__ __forceinline__ float finalize_color(float c) {   // :165 nan_to_num(nan=0,posinf=1,neginf=0).clamp(0,1)
    if (isnan(c)) c = 0.0f;
    return fminf(fmaxf(c, 0.0f), 1.0f);
}

// dL/dcomp of one channel: either handed in (g_comp), or the MSE term of the step's loss formed right here from the
// recomputed composite and the target -- train/trainer.py:999-1004: mse(guard(comp), guard(target)), guard = nan_to_num(nan=0,
// posinf=1, neginf=0).clamp(0,1); loss_scale = 2 * grad_scale / (3 B).  (The composite's own clamp mask is applied by the caller.)
__device__ __forceinline__ float comp_grad(const float* __restrict__ g_comp, const float* __restrict__ target, float loss_scale, float craw,
                                           int64_t i) {
    if (!target) return g_comp ? __ldg(g_comp + i) : 0.0f;             // a missing g_comp counts as zero
    float t = __ldg(target + i);
    if (isnan(t)) t = 0.0f;
    t = fminf(fmaxf(t, 0.0f), 1.0f);
    return (finalize_color(craw) - t) * loss_scale;
}

template <bool RAW>
__global__ void __launch_bounds__(kCompWarps * 32)
composite_fwd_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma,
                     const float* __restrict__ noise, float noise_std, const float* __restrict__ z,
                     const float* __restrict__ ray_norm, float* __restrict__ comp, float* __restrict__ weights,
                     float* __restrict__ acc_out, float* __restrict__ depth_out, int64_t B, int N, uint32_t flags,
                     float eps, uint64_t seed, uint64_t offset, const uint64_t* step_dev, int64_t idx0) {
    if (step_dev) offset += 8 * *step_dev;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    for (int64_t b = blockIdx.x * (int64_t)kCompWarps + warp; b < B; b += (int64_t)gridDim.x * kCompWarps) {
        const float* zrow = z + b * N;
        const bool has_rn = ray_norm != nullptr;
        const float rn = has_rn ? ray_norm[b] : 1.0f;
        float carry = 1.0f, sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            const bool valid = i < N;
            float f = 1.0f, alpha = 0.f, zi = 0.f;
            Sample s = {0.f, 0.f, 0.f, 0.f};
            if (valid) {
                zi = zrow[i];
                s = load_sample<RAW>(rgb_or_raw, sigma, noise, noise_std, add_noise, seed, offset, b * N + i, nullptr, nullptr, softplus, idx0);
                const float sdt = fminf(fmaxf(s.sigma * delta_at(zrow, i, N, inf_last, rn, has_rn), 0.0f), 60.0f);  // :144
                alpha = 1.0f - expf(-sdt);                     // :145
                f = (1.0f - alpha) + eps;                      // :149
            }
            const float incl = warp_scan_mul(f, lane);
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            const float T = carry * excl;                      // :148-150 exclusive cumprod
            carry *= __shfl_sync(0xffffffffu, incl, 31);
            float w = T * alpha;                               // :153
            if (!isfinite(w)) w = 0.0f;                        // :154
            if (valid) {
                if (weights) weights[b * N + i] = w;
                sw += w; swz += w * zi; sr += w * s.r; sg += w * s.g; sb += w * s.b;
            }
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        if (lane == 0) {
            const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);    // :156
            const float bg = white ? (1.0f - acc) : 0.0f;      // :161-162
            comp[b * 3 + 0] = finalize_color(sr + bg);
            comp[b * 3 + 1] = finalize_color(sg + bg);
            comp[b * 3 + 2] = finalize_color(sb + bg);
            if (acc_out) acc_out[b] = acc;
            if (depth_out) depth_out[b] = swz / (acc + eps);   // :157
        }
    }
}

// Backward.  Shared memory per warp: alpha[N], T[N].
template <bool RAW>
__global__ void __launch_bounds__(kCompWarps * 32)
composite_bwd_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma,
                     const float* __restrict__ noise, float noise_std, const float* __restrict__ z,
                     const float* __restrict__ ray_norm, const float* __restrict__ g_comp,
                     const float* __restrict__ g_weights, const float* __restrict__ g_acc,
                     const float* __restrict__ g_depth, float* __restrict__ d_rgb_or_raw, float* __restrict__ d_sigma,
                     int64_t B, int N, uint32_t flags, float eps, uint64_t seed, uint64_t offset, const uint64_t* step_dev,
                     int64_t idx0, const float* __restrict__ target, float loss_scale) {
    if (step_dev) offset += 8 * *step_dev;
    extern __shared__ float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_alpha = smem + (size_t)warp * 3 * N;
    float* s_T = s_alpha + N;
    float* s_pre = s_T + N;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    for (int64_t b = blockIdx.x * (int64_t)kCompWarps + warp; b < B; b += (int64_t)gridDim.x * kCompWarps) {
        const float* zrow = z + b * N;
        const bool has_rn = ray_norm != nullptr;
        const float rn = has_rn ? ray_norm[b] : 1.0f;
        // ---- pass 1: forward recompute, totals
        float carry = 1.0f, sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            const bool valid = i < N;
            float f = 1.0f, alpha = 0.f, zi = 0.f;
            Sample s = {0.f, 0.f, 0.f, 0.f};
            if (valid) {
                zi = zrow[i];
                float pre1 = 0.f;
                s = load_sample<RAW>(rgb_or_raw, sigma, noise, noise_std, add_noise, seed, offset, b * N + i, &pre1, nullptr, softplus, idx0);
                if (RAW) s_pre[i] = pre1;
                const float sdt = fminf(fmaxf(s.sigma * delta_at(zrow, i, N, inf_last, rn, has_rn), 0.0f), 60.0f);
                alpha = 1.0f - expf(-sdt);
                f = (1.0f - alpha) + eps;
            }
            const float incl = warp_scan_mul(f, lane);
            float excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = 1.0f;
            const float T = carry * excl;
            carry *= __shfl_sync(0xffffffffu, incl, 31);
            float w = T * alpha;
            if (!isfinite(w)) w = 0.0f;
            if (valid) {
                s_alpha[i] = alpha; s_T[i] = T;
                sw += w; swz += w * zi; sr += w * s.r; sg += w * s.g; sb += w * s.b;
            }
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        __syncwarp();
        const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);
        const float bg = white ? (1.0f - acc) : 0.0f;
        // clamp/nan_to_num masks on the composite (:165): grad passes on the closed interval, finite only
        float gc[3];
        {
            const float craw[3] = {sr + bg, sg + bg, sb + bg};
#pragma unroll
            for (int c = 0; c < 3; ++c)
                gc[c] = (isfinite(craw[c]) && craw[c] >= 0.0f && craw[c] <= 1.0f) ? comp_grad(g_comp, target, loss_scale, craw[c], b * 3 + c) : 0.0f;
        }
        const float inv = 1.0f / (acc + eps);
        const float gd = g_depth ? g_depth[b] : 0.0f;
        float g_accv = g_acc ? g_acc[b] : 0.0f;
        if (white) g_accv -= gc[0] + gc[1] + gc[2];
        g_accv -= gd * swz * inv * inv;                        // depth = swz/(acc+eps)
        const float g_s = (sw >= 0.0f && sw <= 1.0f) ? g_accv : 0.0f;   // clamp(0,1) mask at :156
        // ---- pass 2: reverse walk with suffix sum of G_i * w_i
        float suffix_carry = 0.0f;
        const int nchunks = (N + 31) / 32;
        for (int ch = nchunks - 1; ch >= 0; --ch) {
            const int i = ch * 32 + lane;
            const bool valid = i < N;
            float Gw = 0.f, G = 0.f, T = 0.f, alpha = 0.f, delta = 0.f, pre = 0.f, w = 0.f;
            Sample s = {0.f, 0.f, 0.f, 0.f};
            if (valid) {
                alpha = s_alpha[i]; T = s_T[i];
                s = load_sample<RAW>(rgb_or_raw, sigma, noise, noise_std, add_noise, seed, offset, b * N + i, &pre, RAW ? &s_pre[i] : nullptr, softplus);
                delta = delta_at(zrow, i, N, inf_last, rn, has_rn);
                const float wraw = T * alpha;
                const bool fin = isfinite(wraw);
                w = fin ? wraw : 0.0f;
                G = (g_weights ? g_weights[b * N + i] : 0.0f) + g_s + s.r * gc[0] + s.g * gc[1] + s.b * gc[2] +
                    gd * zrow[i] * inv;
                if (!fin) G = 0.0f;                            // nan_to_num backward
                Gw = G * w;
            }
            // reverse inclusive scan (suffix within the chunk)
            float sfx = Gw;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float t = __shfl_down_sync(0xffffffffu, sfx, d);
                if (lane + d < 32) sfx += t;
            }
            const float chunk_total = __shfl_sync(0xffffffffu, sfx, 0);
            const float suffix_excl = (sfx - Gw) + suffix_carry;   // sum_{j>i} G_j w_j
            suffix_carry += chunk_total;
            if (valid) {
                const float f = (1.0f - alpha) + eps;
                const float d_alpha = G * T - suffix_excl / f;     // cumprod_backward, division form
                const float d_sdt = d_alpha * (1.0f - alpha);      // d/dsdt (1-exp(-sdt)) = exp(-sdt)
                const float sd = s.sigma * delta;
                float ds = (sd >= 0.0f && sd <= 60.0f) ? d_sdt * delta : 0.0f;   // clamp masks :144
                const int64_t q = b * N + i;
                if (RAW) {
                    float4 o;
                    o.x = w * gc[0] * s.r * (1.0f - s.r);
                    o.y = w * gc[1] * s.g * (1.0f - s.g);
                    o.z = w * gc[2] * s.b * (1.0f - s.b);
                    // relu / softplus backward (softplus: sigmoid(pre), 1 above the threshold)
                    o.w = softplus ? (pre > 20.0f ? ds : ds / (1.0f + expf(-pre))) : (pre > 0.0f ? ds : 0.0f);
                    reinterpret_cast<float4*>(d_rgb_or_raw)[q] = o;
                } else {
                    d_rgb_or_raw[q * 3 + 0] = w * gc[0];
                    d_rgb_or_raw[q * 3 + 1] = w * gc[1];
                    d_rgb_or_raw[q * 3 + 2] = w * gc[2];
                    d_sigma[q] = ds;
                }
            }
        }
        __syncwarp();
    }
}

// =====================================================================================================================
// Run layout (N <= 192 samples per ray -- every vanilla shape: 64 coarse, 192 merged; 192 < N <= 1024: the multi-warp variant
// further down): lane l of the ray's warp owns the
// CONTIGUOUS run [l R, l R + R) of samples, R = ceil(N / 32) <= 8, all in registers.  The exclusive cumprod is a serial
// product inside the run plus ONE multiplicative warp scan over the 32 run products per ray (instead of one scan per 32
// samples), the loads of a run are issued up front (R independent 16-byte loads per lane in flight), and the backward keeps
// alpha / T / rgb / pre-activations of its run in registers between the two passes: no shared memory, no recompute of the
// activations.  Head activations use MUFU-based fast paths (ex2 / rcp: relative error ~2e-7, far inside the 1e-4 bar).
// The strided kernels above remain for N > 1024.
// =====================================================================================================================
constexpr int kRunWarps = 4;
// One warp per ray up to 192 samples (R <= 6); above, 2-4 warps per ray with R = 4..6 each (7, 8 beyond 768): measured, the R = 8
// single-warp kernels (120-160 registers) stream at 0.53-0.58 of the HBM roof where R <= 6 reaches 0.7-0.86.
constexpr int kRunOneWarpMaxN = 192;
constexpr int kRunMaxN = 1024;                  // up to 4 warps per ray

// 1 / (1 + 2^(-x log2 e)): FMUL + MUFU.EX2 + FADD + MUFU.RCP (relative error ~4e-7; saturates to 0 / 1, NaN propagates)
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }

template <bool RAW, int R>
struct RunSamples {
    float r[R], g[R], b[R], sigma[R], pre[R], z[R], delta[R], alpha[R], Tl[R];
};

// Loads + activations + alpha + in-run exclusive products for this lane's run; returns the run's product of (1 - alpha + eps).
// FULL: N == 32 R, every lane owns exactly R samples (64 / 192 / 256 samples per ray): no per-sample validity predicates.
// In-kernel noise is drawn in pairs (one hash + Box-Muller -> cos and sin branches) for samples (k, k+1) of the run, k even;
// forward and backward call this same function, so they regenerate identical draws.
template <bool RAW, int R, bool FULL>
__device__ __forceinline__ float run_forward(RunSamples<RAW, R>& s, const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma,
                                             const float* __restrict__ noise, float noise_std, bool add_noise, bool softplus,
                                             uint64_t seed, uint64_t offset, const float* __restrict__ zrow, int64_t q0, int start, int cnt,
                                             int N, bool inf_last, float rn, bool has_rn, float eps, int64_t idx0, bool multi_warp = false) {
    float4 v[R];
    float nz[R];
#pragma unroll
    for (int k = 0; k < R; ++k) {              // every load of the run in flight before the first use
        s.z[k] = 0.f; nz[k] = 0.f; v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (FULL || k < cnt) {
            s.z[k] = __ldg(zrow + start + k);
            if (RAW) {
                v[k] = __ldg(reinterpret_cast<const float4*>(rgb_or_raw) + q0 + k);
                if (add_noise && noise) nz[k] = __ldg(noise + q0 + k);
            } else {
                v[k].x = __ldg(rgb_or_raw + (q0 + k) * 3); v[k].y = __ldg(rgb_or_raw + (q0 + k) * 3 + 1);
                v[k].z = __ldg(rgb_or_raw + (q0 + k) * 3 + 2); v[k].w = __ldg(sigma + q0 + k);
            }
        }
    }
    float z_next_lane = __shfl_down_sync(0xffffffffu, s.z[0], 1);            // first z of the next lane's run
    if (multi_warp && (threadIdx.x & 31) == 31 && start + R < N) z_next_lane = __ldg(zrow + start + R);   // ... which the next WARP owns
    if (RAW && add_noise && !noise) {
        const uint32_t key = hash_key(seed, offset, (uint64_t)(q0 + idx0));
#pragma unroll
        for (int k = 0; k < R; k += 2) {
            float n0, n1;
            hash_normal_pair(key, (uint32_t)(q0 + idx0 + k), n0, n1);
            nz[k] = n0;
            if (k + 1 < R) nz[k + 1] = n1;
        }
    }
    float prod = 1.0f;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        s.alpha[k] = 0.f; s.Tl[k] = prod; s.r[k] = s.g[k] = s.b[k] = s.sigma[k] = s.pre[k] = s.delta[k] = 0.f;
        if (FULL || k < cnt) {
            if (RAW) {
                s.r[k] = fast_sigmoid(v[k].x); s.g[k] = fast_sigmoid(v[k].y); s.b[k] = fast_sigmoid(v[k].z);       // :236
                float pre = v[k].w;
                if (add_noise) pre = fmaf(nz[k], noise_std, pre);                                                   // :239-241
                s.pre[k] = pre;
                s.sigma[k] = softplus ? (pre > 20.0f ? pre : log1pf(__expf(pre))) : fmaxf(pre, 0.0f);              // :243-246
            } else {
                s.r[k] = v[k].x; s.g[k] = v[k].y; s.b[k] = v[k].z; s.sigma[k] = v[k].w;
            }
            const int i = start + k;
            float zn = z_next_lane;
            if (k + 1 < R) zn = (FULL || k + 1 < cnt) ? s.z[k + 1] : z_next_lane;
            float d = (i == N - 1) ? (inf_last ? 1e10f : 0.0f) : (zn - s.z[k]);                                    // :131-136
            if (has_rn) d *= rn;                                                                                   // :139-141
            s.delta[k] = d;
            const float sdt = fminf(fmaxf(s.sigma[k] * d, 0.0f), 60.0f);                                           // :144
            // :145 -- the accurate expf: for small sigma*delta, alpha inherits the ABSOLUTE error of exp (a 2^-22 MUFU error is a
            // 1e-4 relative error of alpha = 1e-3), which is what the 1e-4 parity bar on the composite cannot afford
            s.alpha[k] = 1.0f - expf(-sdt);
            prod *= (1.0f - s.alpha[k]) + eps;                                                                     // :149
        }
    }
    return prod;
}

template <bool RAW, int R, bool FULL>
__global__ void __launch_bounds__(kRunWarps * 32)
composite_fwd_run_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma, const float* __restrict__ noise,
                         float noise_std, const float* __restrict__ z, const float* __restrict__ ray_norm, float* __restrict__ comp,
                         float* __restrict__ weights, float* __restrict__ acc_out, float* __restrict__ depth_out, int64_t B, int N,
                         uint32_t flags, float eps, uint64_t seed, uint64_t offset, const uint64_t* step_dev, int64_t idx0) {
    if (step_dev) offset += 8 * *step_dev;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    const bool has_rn = ray_norm != nullptr;
    const int start = lane * R;
    const int cnt = FULL ? R : max(0, min(R, N - start));
    for (int64_t b = blockIdx.x * (int64_t)kRunWarps + warp; b < B; b += (int64_t)gridDim.x * kRunWarps) {
        const float rn = has_rn ? __ldg(ray_norm + b) : 1.0f;
        const int64_t q0 = b * N + start;
        RunSamples<RAW, R> s;
        const float prod = run_forward<RAW, R, FULL>(s, rgb_or_raw, sigma, noise, noise_std, add_noise, softplus, seed, offset, z + b * N, q0, start,
                                               cnt, N, inf_last, rn, has_rn, eps, idx0);
        const float incl = warp_scan_mul(prod, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);                   // product over all earlier lanes' runs
        if (lane == 0) excl = 1.0f;
        float sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            if (FULL || k < cnt) {
                float w = (excl * s.Tl[k]) * s.alpha[k];                     // :148-153 exclusive cumprod, weights
                if (!isfinite(w)) w = 0.0f;                                  // :154
                if (weights) weights[q0 + k] = w;
                sw += w; swz = fmaf(w, s.z[k], swz); sr = fmaf(w, s.r[k], sr); sg = fmaf(w, s.g[k], sg); sb = fmaf(w, s.b[k], sb);
            }
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        if (lane == 0) {
            const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);                  // :156
            const float bg = white ? (1.0f - acc) : 0.0f;                    // :161-162
            comp[b * 3 + 0] = finalize_color(sr + bg);
            comp[b * 3 + 1] = finalize_color(sg + bg);
            comp[b * 3 + 2] = finalize_color(sb + bg);
            if (acc_out) acc_out[b] = acc;
            if (depth_out) depth_out[b] = swz / (acc + eps);                 // :157
        }
    }
}

template <bool RAW, int R, bool FULL>
__global__ void __launch_bounds__(kRunWarps * 32)
composite_bwd_run_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma, const float* __restrict__ noise,
                         float noise_std, const float* __restrict__ z, const float* __restrict__ ray_norm, const float* __restrict__ g_comp,
                         const float* __restrict__ g_weights, const float* __restrict__ g_acc, const float* __restrict__ g_depth,
                         float* __restrict__ d_rgb_or_raw, float* __restrict__ d_sigma, int64_t B, int N, uint32_t flags, float eps,
                         uint64_t seed, uint64_t offset, const uint64_t* step_dev, int64_t idx0, const float* __restrict__ target,
                         float loss_scale) {
    if (step_dev) offset += 8 * *step_dev;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    const bool has_rn = ray_norm != nullptr;
    const int start = lane * R;
    const int cnt = FULL ? R : max(0, min(R, N - start));
    for (int64_t b = blockIdx.x * (int64_t)kRunWarps + warp; b < B; b += (int64_t)gridDim.x * kRunWarps) {
        const float rn = has_rn ? __ldg(ray_norm + b) : 1.0f;
        const int64_t q0 = b * N + start;
        // ---- pass 1: forward recompute, everything about this lane's run stays in registers
        RunSamples<RAW, R> s;
        const float prod = run_forward<RAW, R, FULL>(s, rgb_or_raw, sigma, noise, noise_std, add_noise, softplus, seed, offset, z + b * N, q0, start,
                                               cnt, N, inf_last, rn, has_rn, eps, idx0);
        float gwv[R];
#pragma unroll
        for (int k = 0; k < R; ++k) gwv[k] = (g_weights && (FULL || k < cnt)) ? __ldg(g_weights + q0 + k) : 0.0f;
        const float incl = warp_scan_mul(prod, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.0f;
        float sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
        float T[R], w[R];
        bool fin[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            T[k] = excl * s.Tl[k];
            const float wraw = T[k] * s.alpha[k];
            fin[k] = isfinite(wraw);
            w[k] = ((FULL || k < cnt) && fin[k]) ? wraw : 0.0f;
            sw += w[k]; swz = fmaf(w[k], s.z[k], swz); sr = fmaf(w[k], s.r[k], sr); sg = fmaf(w[k], s.g[k], sg); sb = fmaf(w[k], s.b[k], sb);
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);
        const float bg = white ? (1.0f - acc) : 0.0f;
        float gc[3];                                   // clamp / nan_to_num masks on the composite (:165)
        {
            const float craw[3] = {sr + bg, sg + bg, sb + bg};
#pragma unroll
            for (int c = 0; c < 3; ++c)
                gc[c] = (isfinite(craw[c]) && craw[c] >= 0.0f && craw[c] <= 1.0f) ? comp_grad(g_comp, target, loss_scale, craw[c], b * 3 + c) : 0.0f;
        }
        const float inv = 1.0f / (acc + eps);
        const float gd = g_depth ? __ldg(g_depth + b) : 0.0f;
        float g_accv = g_acc ? __ldg(g_acc + b) : 0.0f;
        if (white) g_accv -= gc[0] + gc[1] + gc[2];
        g_accv -= gd * swz * inv * inv;                                      // depth = swz / (acc + eps)
        const float g_s = (sw >= 0.0f && sw <= 1.0f) ? g_accv : 0.0f;        // clamp(0,1) mask at :156
        // ---- pass 2: G_i, suffix sums of G_j w_j (serial inside the run + one reverse warp scan per ray)
        float G[R], lane_total = 0.f;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            G[k] = 0.f;
            if ((FULL || k < cnt) && fin[k])                                 // (nan_to_num backward: no gradient through a non-finite weight)
                G[k] = gwv[k] + g_s + s.r[k] * gc[0] + s.g[k] * gc[1] + s.b[k] * gc[2] + gd * s.z[k] * inv;
            lane_total = fmaf(G[k], w[k], lane_total);
        }
        float sfx = lane_total;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const float t = __shfl_down_sync(0xffffffffu, sfx, d);
            if (lane + d < 32) sfx += t;
        }
        float suffix = sfx - lane_total;                                     // sum over all later lanes' runs
#pragma unroll
        for (int k = R - 1; k >= 0; --k) {
            if (FULL || k < cnt) {
                const float f = (1.0f - s.alpha[k]) + eps;
                const float d_alpha = G[k] * T[k] - suffix * rcp_approx(f);  // cumprod_backward, division form (f in [1e-10, 1])
                suffix = fmaf(G[k], w[k], suffix);
                const float d_sdt = d_alpha * (1.0f - s.alpha[k]);           // d/dsdt (1 - exp(-sdt)) = exp(-sdt)
                const float sd = s.sigma[k] * s.delta[k];
                const float ds = (sd >= 0.0f && sd <= 60.0f) ? d_sdt * s.delta[k] : 0.0f;     // clamp masks :144
                if (RAW) {
                    float4 o;
                    o.x = w[k] * gc[0] * s.r[k] * (1.0f - s.r[k]);
                    o.y = w[k] * gc[1] * s.g[k] * (1.0f - s.g[k]);
                    o.z = w[k] * gc[2] * s.b[k] * (1.0f - s.b[k]);
                    o.w = softplus ? (s.pre[k] > 20.0f ? ds : ds * fast_sigmoid(s.pre[k])) : (s.pre[k] > 0.0f ? ds : 0.0f);
                    reinterpret_cast<float4*>(d_rgb_or_raw)[q0 + k] = o;
                } else {
                    d_rgb_or_raw[(q0 + k) * 3 + 0] = w[k] * gc[0];
                    d_rgb_or_raw[(q0 + k) * 3 + 1] = w[k] * gc[1];
                    d_rgb_or_raw[(q0 + k) * 3 + 2] = w[k] * gc[2];
                    d_sigma[q0 + k] = ds;
                }
            }
        }
    }
}

// ---- 192 < N <= 1024: the same run layout with W = 2..4 warps per ray (one block = one ray at a time).  Warp w owns
// samples [32 R w, 32 R (w + 1)) with R = ceil(N / (32 W)) per lane (an even split: no warp is left with a stub); transmittance is multiplicative, so each warp works relative to its own
// first sample and the products of the earlier warps' segments (exchanged through shared memory) scale it afterwards; the
// per-ray sums and the backward's suffix sums are combined the same way.  No serial pass over the ray, same registers.
template <bool RAW, int W, int R>
__global__ void __launch_bounds__(W * 32)
composite_fwd_runw_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma, const float* __restrict__ noise,
                          float noise_std, const float* __restrict__ z, const float* __restrict__ ray_norm, float* __restrict__ comp,
                          float* __restrict__ weights, float* __restrict__ acc_out, float* __restrict__ depth_out, int64_t B, int N,
                          uint32_t flags, float eps, uint64_t seed, uint64_t offset, const uint64_t* step_dev, int64_t idx0) {
    if (step_dev) offset += 8 * *step_dev;
    __shared__ float s_prod[2][W], s_sum[2][W][5];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    const bool has_rn = ray_norm != nullptr;
    const int start = warp * 32 * R + lane * R;
    const int cnt = max(0, min(R, N - start));
    int par = 0;
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x, par ^= 1) {
        const float rn = has_rn ? __ldg(ray_norm + b) : 1.0f;
        const int64_t q0 = b * N + start;
        RunSamples<RAW, R> s;
        const float prod = run_forward<RAW, R, false>(s, rgb_or_raw, sigma, noise, noise_std, add_noise, softplus, seed, offset, z + b * N, q0, start,
                                                cnt, N, inf_last, rn, has_rn, eps, idx0, true);
        const float incl = warp_scan_mul(prod, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.0f;
        if (lane == 31) s_prod[par][warp] = incl;
        __syncthreads();
        float carry = 1.0f;                                                  // product over the earlier warps' segments
#pragma unroll
        for (int v = 0; v < W; ++v) if (v < warp) carry *= s_prod[par][v];
        excl *= carry;
        float sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            if (k < cnt) {
                float w = (excl * s.Tl[k]) * s.alpha[k];
                if (!isfinite(w)) w = 0.0f;
                if (weights) weights[q0 + k] = w;
                sw += w; swz = fmaf(w, s.z[k], swz); sr = fmaf(w, s.r[k], sr); sg = fmaf(w, s.g[k], sg); sb = fmaf(w, s.b[k], sb);
            }
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        if (lane == 0) { s_sum[par][warp][0] = sw; s_sum[par][warp][1] = swz; s_sum[par][warp][2] = sr; s_sum[par][warp][3] = sg; s_sum[par][warp][4] = sb; }
        __syncthreads();
        if (threadIdx.x == 0) {
            sw = swz = sr = sg = sb = 0.f;
#pragma unroll
            for (int v = 0; v < W; ++v) { sw += s_sum[par][v][0]; swz += s_sum[par][v][1]; sr += s_sum[par][v][2]; sg += s_sum[par][v][3]; sb += s_sum[par][v][4]; }
            const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);
            const float bg = white ? (1.0f - acc) : 0.0f;
            comp[b * 3 + 0] = finalize_color(sr + bg);
            comp[b * 3 + 1] = finalize_color(sg + bg);
            comp[b * 3 + 2] = finalize_color(sb + bg);
            if (acc_out) acc_out[b] = acc;
            if (depth_out) depth_out[b] = swz / (acc + eps);
        }
    }
}

template <bool RAW, int W, int R>
__global__ void __launch_bounds__(W * 32)
composite_bwd_runw_kernel(const float* __restrict__ rgb_or_raw, const float* __restrict__ sigma, const float* __restrict__ noise,
                          float noise_std, const float* __restrict__ z, const float* __restrict__ ray_norm, const float* __restrict__ g_comp,
                          const float* __restrict__ g_weights, const float* __restrict__ g_acc, const float* __restrict__ g_depth,
                          float* __restrict__ d_rgb_or_raw, float* __restrict__ d_sigma, int64_t B, int N, uint32_t flags, float eps,
                          uint64_t seed, uint64_t offset, const uint64_t* step_dev, int64_t idx0, const float* __restrict__ target,
                          float loss_scale) {
    if (step_dev) offset += 8 * *step_dev;
    __shared__ float s_prod[2][W], s_sum[2][W][5], s_tot[2][W];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool white = flags & NSB_WHITE_BKGD, inf_last = flags & NSB_INFINITE_LAST_BIN;
    const bool add_noise = RAW && (flags & NSB_TRAINING) && noise_std > 0.0f;
    const bool softplus = RAW && (flags & NSB_SIGMA_SOFTPLUS);
    const bool has_rn = ray_norm != nullptr;
    const int start = warp * 32 * R + lane * R;
    const int cnt = max(0, min(R, N - start));
    int par = 0;
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x, par ^= 1) {
        const float rn = has_rn ? __ldg(ray_norm + b) : 1.0f;
        const int64_t q0 = b * N + start;
        RunSamples<RAW, R> s;
        const float prod = run_forward<RAW, R, false>(s, rgb_or_raw, sigma, noise, noise_std, add_noise, softplus, seed, offset, z + b * N, q0, start,
                                                cnt, N, inf_last, rn, has_rn, eps, idx0, true);
        float gwv[R];
#pragma unroll
        for (int k = 0; k < R; ++k) gwv[k] = (g_weights && k < cnt) ? __ldg(g_weights + q0 + k) : 0.0f;
        const float incl = warp_scan_mul(prod, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.0f;
        if (lane == 31) s_prod[par][warp] = incl;
        __syncthreads();
        float carry = 1.0f;
#pragma unroll
        for (int v = 0; v < W; ++v) if (v < warp) carry *= s_prod[par][v];
        excl *= carry;
        float sw = 0.f, swz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
        float T[R], w[R];
        bool fin[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            T[k] = excl * s.Tl[k];
            const float wraw = T[k] * s.alpha[k];
            fin[k] = isfinite(wraw);
            w[k] = (k < cnt && fin[k]) ? wraw : 0.0f;
            sw += w[k]; swz = fmaf(w[k], s.z[k], swz); sr = fmaf(w[k], s.r[k], sr); sg = fmaf(w[k], s.g[k], sg); sb = fmaf(w[k], s.b[k], sb);
        }
        sw = warp_sum(sw); swz = warp_sum(swz); sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
        if (lane == 0) { s_sum[par][warp][0] = sw; s_sum[par][warp][1] = swz; s_sum[par][warp][2] = sr; s_sum[par][warp][3] = sg; s_sum[par][warp][4] = sb; }
        __syncthreads();
        sw = swz = sr = sg = sb = 0.f;                                       // every thread: the ray's totals, same order in every thread
#pragma unroll
        for (int v = 0; v < W; ++v) { sw += s_sum[par][v][0]; swz += s_sum[par][v][1]; sr += s_sum[par][v][2]; sg += s_sum[par][v][3]; sb += s_sum[par][v][4]; }
        const float acc = fminf(fmaxf(sw, 0.0f), 1.0f);
        const float bg = white ? (1.0f - acc) : 0.0f;
        float gc[3];
        {
            const float craw[3] = {sr + bg, sg + bg, sb + bg};
#pragma unroll
            for (int c = 0; c < 3; ++c)
                gc[c] = (isfinite(craw[c]) && craw[c] >= 0.0f && craw[c] <= 1.0f) ? comp_grad(g_comp, target, loss_scale, craw[c], b * 3 + c) : 0.0f;
        }
        const float inv = 1.0f / (acc + eps);
        const float gd = g_depth ? __ldg(g_depth + b) : 0.0f;
        float g_accv = g_acc ? __ldg(g_acc + b) : 0.0f;
        if (white) g_accv -= gc[0] + gc[1] + gc[2];
        g_accv -= gd * swz * inv * inv;
        const float g_s = (sw >= 0.0f && sw <= 1.0f) ? g_accv : 0.0f;
        float G[R], lane_total = 0.f;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            G[k] = 0.f;
            if (k < cnt && fin[k]) G[k] = gwv[k] + g_s + s.r[k] * gc[0] + s.g[k] * gc[1] + s.b[k] * gc[2] + gd * s.z[k] * inv;
            lane_total = fmaf(G[k], w[k], lane_total);
        }
        float sfx = lane_total;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const float t = __shfl_down_sync(0xffffffffu, sfx, d);
            if (lane + d < 32) sfx += t;
        }
        if (lane == 0) s_tot[par][warp] = sfx;                               // this warp's segment total of G w
        __syncthreads();
        float suffix = sfx - lane_total;                                     // later lanes of this warp ...
#pragma unroll
        for (int v = 0; v < W; ++v) if (v > warp) suffix += s_tot[par][v];   // ... and the later warps' segments
#pragma unroll
        for (int k = R - 1; k >= 0; --k) {
            if (k < cnt) {
                const float f = (1.0f - s.alpha[k]) + eps;
                const float d_alpha = G[k] * T[k] - suffix * rcp_approx(f);
                suffix = fmaf(G[k], w[k], suffix);
                const float d_sdt = d_alpha * (1.0f - s.alpha[k]);
                const float sd = s.sigma[k] * s.delta[k];
                const float ds = (sd >= 0.0f && sd <= 60.0f) ? d_sdt * s.delta[k] : 0.0f;
                if (RAW) {
                    float4 o;
                    o.x = w[k] * gc[0] * s.r[k] * (1.0f - s.r[k]);
                    o.y = w[k] * gc[1] * s.g[k] * (1.0f - s.g[k]);
                    o.z = w[k] * gc[2] * s.b[k] * (1.0f - s.b[k]);
                    o.w = softplus ? (s.pre[k] > 20.0f ? ds : ds * fast_sigmoid(s.pre[k])) : (s.pre[k] > 0.0f ? ds : 0.0f);
                    reinterpret_cast<float4*>(d_rgb_or_raw)[q0 + k] = o;
                } else {
                    d_rgb_or_raw[(q0 + k) * 3 + 0] = w[k] * gc[0];
                    d_rgb_or_raw[(q0 + k) * 3 + 1] = w[k] * gc[1];
                    d_rgb_or_raw[(q0 + k) * 3 + 2] = w[k] * gc[2];
                    d_sigma[q0 + k] = ds;
                }
            }
        }
    }
}

static int runw_grid(int64_t B, int W) {
    const int64_t cap = (int64_t)num_sms() * (64 / W);       // up to 64 warps per SM
    return (int)(B < cap ? (B > 0 ? B : 1) : cap);
}

static int run_grid(int64_t B) {
    const int64_t want = cdiv(B, kRunWarps);
    const int64_t cap = (int64_t)num_sms() * 32;
    return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

template <bool RAW>
static int launch_fwd_run(const float* a, const float* sigma, const float* noise, float noise_std, const float* z, const float* rn,
                          float* comp, float* weights, float* acc, float* depth, int64_t B, int N, uint32_t flags, float eps, uint64_t seed,
                          uint64_t off, void* stream, int64_t idx0 = 0) {
    const int R = (N + 31) / 32;
    cudaStream_t st = as_stream(stream);
    if (N > kRunOneWarpMaxN) {
        const int W = N <= 768 ? (N + 191) / 192 : 4, RW = (N + 32 * W - 1) / (32 * W), gridw = runw_grid(B, W);
#define NSB_RUNW_FWD(WW, RR) \
        else if (W == WW && RW == RR) composite_fwd_runw_kernel<RAW, WW, RR><<<gridw, WW * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, comp, weights, acc, depth, B, N, flags, eps, seed, off, g_step_dev, idx0);
        if (false) {}
        NSB_RUNW_FWD(2, 4) NSB_RUNW_FWD(2, 5) NSB_RUNW_FWD(2, 6)
        NSB_RUNW_FWD(3, 5) NSB_RUNW_FWD(3, 6)
        NSB_RUNW_FWD(4, 5) NSB_RUNW_FWD(4, 6) NSB_RUNW_FWD(4, 7) NSB_RUNW_FWD(4, 8)
        else return NSB_E_BADARG;
#undef NSB_RUNW_FWD
        NSB_LAUNCH_CHECK("composite_fwd_runw_kernel");
        return NSB_OK;
    }
    const int grid = run_grid(B);
#define NSB_RUN_FWD(RR)                                                                                                              \
    case RR:                                                                                                                         \
        if (N == 32 * RR) composite_fwd_run_kernel<RAW, RR, true><<<grid, kRunWarps * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, comp, weights, \
                                                                                                    acc, depth, B, N, flags, eps, seed, off, g_step_dev, idx0); \
        else composite_fwd_run_kernel<RAW, RR, false><<<grid, kRunWarps * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, comp, weights, acc, depth, \
                                                                                        B, N, flags, eps, seed, off, g_step_dev, idx0);           \
        break;
    switch (R) { NSB_RUN_FWD(1) NSB_RUN_FWD(2) NSB_RUN_FWD(3) NSB_RUN_FWD(4) NSB_RUN_FWD(5) NSB_RUN_FWD(6) NSB_RUN_FWD(7) NSB_RUN_FWD(8)
        default: return NSB_E_BADARG; }
#undef NSB_RUN_FWD
    NSB_LAUNCH_CHECK("composite_fwd_run_kernel");
    return NSB_OK;
}

template <bool RAW>
static int launch_bwd_run(const float* a, const float* sigma, const float* noise, float noise_std, const float* z, const float* rn,
                          const float* g_comp, const float* g_w, const float* g_a, const float* g_d, float* d0, float* d1, int64_t B, int N,
                          uint32_t flags, float eps, uint64_t seed, uint64_t off, void* stream, int64_t idx0 = 0, const float* target = nullptr,
                          float loss_scale = 0.f) {
    const int R = (N + 31) / 32;
    cudaStream_t st = as_stream(stream);
    if (N > kRunOneWarpMaxN) {
        const int W = N <= 768 ? (N + 191) / 192 : 4, RW = (N + 32 * W - 1) / (32 * W), gridw = runw_grid(B, W);
#define NSB_RUNW_BWD(WW, RR) \
        else if (W == WW && RW == RR) composite_bwd_runw_kernel<RAW, WW, RR><<<gridw, WW * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, g_comp, g_w, g_a, g_d, d0, d1, B, N, flags, eps, seed, off, g_step_dev, idx0, target, loss_scale);
        if (false) {}
        NSB_RUNW_BWD(2, 4) NSB_RUNW_BWD(2, 5) NSB_RUNW_BWD(2, 6)
        NSB_RUNW_BWD(3, 5) NSB_RUNW_BWD(3, 6)
        NSB_RUNW_BWD(4, 5) NSB_RUNW_BWD(4, 6) NSB_RUNW_BWD(4, 7) NSB_RUNW_BWD(4, 8)
        else return NSB_E_BADARG;
#undef NSB_RUNW_BWD
        NSB_LAUNCH_CHECK("composite_bwd_runw_kernel");
        return NSB_OK;
    }
    const int grid = run_grid(B);
#define NSB_RUN_BWD(RR)                                                                                                             \
    case RR:                                                                                                                         \
        if (N == 32 * RR) composite_bwd_run_kernel<RAW, RR, true><<<grid, kRunWarps * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, g_comp, g_w, g_a, \
                                                                                                    g_d, d0, d1, B, N, flags, eps, seed, off, g_step_dev, idx0, target, loss_scale); \
        else composite_bwd_run_kernel<RAW, RR, false><<<grid, kRunWarps * 32, 0, st>>>(a, sigma, noise, noise_std, z, rn, g_comp, g_w, g_a, g_d, d0, d1, \
                                                                                        B, N, flags, eps, seed, off, g_step_dev, idx0, target, loss_scale); \
        break;
    switch (R) { NSB_RUN_BWD(1) NSB_RUN_BWD(2) NSB_RUN_BWD(3) NSB_RUN_BWD(4) NSB_RUN_BWD(5) NSB_RUN_BWD(6) NSB_RUN_BWD(7) NSB_RUN_BWD(8)
        default: return NSB_E_BADARG; }
#undef NSB_RUN_BWD
    NSB_LAUNCH_CHECK("composite_bwd_run_kernel");
    return NSB_OK;
}

static int comp_grid(int64_t B) {
    const int64_t want = cdiv(B, kCompWarps);
    const int64_t cap = (int64_t)num_sms() * 16;
    return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

template <bool RAW>
static int launch_bwd(const float* a, const float* sigma, const float* noise, float noise_std, const float* z,
                      const float* rn, const float* g_comp, const float* g_w, const float* g_a, const float* g_d,
                      float* d0, float* d1, int64_t B, int N, uint32_t flags, float eps, uint64_t seed, uint64_t off,
                      void* stream, int64_t idx0 = 0, const float* target = nullptr, float loss_scale = 0.f) {
    const size_t smem = (size_t)kCompWarps * 3 * N * sizeof(float);
    if (smem > 200 * 1024) return NSB_E_BADARG;
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(composite_bwd_kernel<RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    composite_bwd_kernel<RAW><<<comp_grid(B), kCompWarps * 32, smem, as_stream(stream)>>>(
        a, sigma, noise, noise_std, z, rn, g_comp, g_w, g_a, g_d, d0, d1, B, N, flags, eps, seed, off, g_step_dev, idx0, target, loss_scale);
    NSB_LAUNCH_CHECK("composite_bwd_kernel");
    return NSB_OK;
}

// ---- loss -- train/trainer.py:999-1006 ------------------------------------------------------------
__device__ __forceinline__ float guard01(float x, bool* pass) {   // nan_to_num(nan=0,posinf=1,neginf=0).clamp(0,1)
    *pass = isfinite(x) && x >= 0.0f && x <= 1.0f;
    if (isnan(x)) x = 0.0f;
    return fminf(fmaxf(x, 0.0f), 1.0f);
}

__global__ void mse_zero_kernel(float* scalars) { if (threadIdx.x < 4) scalars[threadIdx.x] = 0.0f; }

__global__ void mse_loss_kernel(const float* __restrict__ comp_c, const float* __restrict__ comp_f,
                                const float* __restrict__ target, float* __restrict__ g_c, float* __restrict__ g_f,
                                float* __restrict__ scalars, int64_t n, float grad_scale) {
    float sc = 0.f, sf = 0.f;
    const float inv_n = 1.0f / (float)n;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        bool pt, pc, pf;
        const float t = guard01(target[i], &pt);
        if (comp_c) {
            const float c = guard01(comp_c[i], &pc);
            const float d = c - t; sc += d * d;
            if (g_c) g_c[i] = pc ? 2.0f * d * inv_n * grad_scale : 0.0f;
        }
        const float f = guard01(comp_f[i], &pf);
        const float d = f - t; sf += d * d;
        if (g_f) g_f[i] = pf ? 2.0f * d * inv_n * grad_scale : 0.0f;
    }
    sc = warp_sum(sc); sf = warp_sum(sf);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&scalars[2], sc * inv_n); atomicAdd(&scalars[3], sf * inv_n); }
}

// small batches (the training step: 3 x 1024 values): one block does zero + reduce + finish, deterministically
__global__ void __launch_bounds__(256) mse_single_block_kernel(const float* __restrict__ comp_c, const float* __restrict__ comp_f,
                                                               const float* __restrict__ target, float* __restrict__ g_c,
                                                               float* __restrict__ g_f, float* __restrict__ scalars, int64_t n,
                                                               float grad_scale) {
    __shared__ float s_c[8], s_f[8];
    float sc = 0.f, sf = 0.f;
    const float inv_n = 1.0f / (float)n;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        bool pt, pc, pf;
        const float t = guard01(target[i], &pt);
        if (comp_c) {
            const float c = guard01(comp_c[i], &pc);
            const float d = c - t; sc += d * d;
            if (g_c) g_c[i] = pc ? 2.0f * d * inv_n * grad_scale : 0.0f;
        }
        const float f = guard01(comp_f[i], &pf);
        const float d = f - t; sf += d * d;
        if (g_f) g_f[i] = pf ? 2.0f * d * inv_n * grad_scale : 0.0f;
    }
    sc = warp_sum(sc); sf = warp_sum(sf);
    if ((threadIdx.x & 31) == 0) { s_c[threadIdx.x >> 5] = sc; s_f[threadIdx.x >> 5] = sf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float mc = 0.f, mf = 0.f;
        for (int w = 0; w < 8; ++w) { mc += s_c[w]; mf += s_f[w]; }
        mc *= inv_n; mf *= inv_n;
        scalars[2] = mc; scalars[3] = mf;
        scalars[0] = mc + mf;                                              // :1005
        scalars[1] = -10.0f * log10f(fmaxf(mf, 1e-10f));                   // trainer.py:77-78
    }
}

__global__ void mse_finish_kernel(float* scalars) {
    if (threadIdx.x == 0) {
        scalars[0] = scalars[2] + scalars[3];                              // :1005
        scalars[1] = -10.0f * log10f(fmaxf(scalars[3], 1e-10f));           // trainer.py:77-78
    }
}

}  // namespace nsb

using namespace nsb;

extern "C" int nsb_composite_fwd(const float* rgb, const float* sigma, const float* z, const float* ray_norm,
                                 float* comp, float* weights, float* acc, float* depth, int64_t B, int N,
                                 uint32_t flags, float eps, void* stream) {
    if (B == 0) return NSB_OK;
    if (!rgb || !sigma || !z || !comp || N < 1 || B < 0) return NSB_E_BADARG;
    if (N <= kRunMaxN) return launch_fwd_run<false>(rgb, sigma, nullptr, 0.f, z, ray_norm, comp, weights, acc, depth, B, N, flags, eps, 0, 0, stream);
    composite_fwd_kernel<false><<<comp_grid(B), kCompWarps * 32, 0, as_stream(stream)>>>(
        rgb, sigma, nullptr, 0.f, z, ray_norm, comp, weights, acc, depth, B, N, flags, eps, 0, 0, nullptr, 0);
    NSB_LAUNCH_CHECK("composite_fwd_kernel");
    return NSB_OK;
}

extern "C" int nsb_composite_bwd(const float* rgb, const float* sigma, const float* z, const float* ray_norm,
                                 const float* g_comp, const float* g_weights, const float* g_acc, const float* g_depth,
                                 float* d_rgb, float* d_sigma, int64_t B, int N, uint32_t flags, float eps,
                                 void* stream) {
    if (B == 0) return NSB_OK;
    if (!rgb || !sigma || !z || !g_comp || !d_rgb || !d_sigma || N < 1 || B < 0) return NSB_E_BADARG;
    if (N <= kRunMaxN)
        return launch_bwd_run<false>(rgb, sigma, nullptr, 0.f, z, ray_norm, g_comp, g_weights, g_acc, g_depth, d_rgb, d_sigma, B, N, flags, eps,
                                     0, 0, stream);
    return launch_bwd<false>(rgb, sigma, nullptr, 0.f, z, ray_norm, g_comp, g_weights, g_acc, g_depth, d_rgb, d_sigma,
                             B, N, flags, eps, 0, 0, stream);
}

namespace nsb {
// nsb_composite_raw_fwd on rays [b0, b0 + B) of a larger batch: idx0 = b0 * N shifts the index of the in-kernel noise draws, so
// a batch processed in pieces draws the same numbers as the batch processed whole (engine.cu: half batches on two streams)
int composite_raw_fwd_at(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm, float* comp,
                         float* weights, float* acc, float* depth, int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset,
                         int64_t idx0, void* stream) {
    if (B == 0) return NSB_OK;
    if (!raw || !z || !comp || N < 1 || B < 0) return NSB_E_BADARG;
    if (N <= kRunMaxN)
        return launch_fwd_run<true>(raw, nullptr, noise, noise_std, z, ray_norm, comp, weights, acc, depth, B, N, flags, 1e-10f, seed, offset, stream,
                                    idx0);
    composite_fwd_kernel<true><<<comp_grid(B), kCompWarps * 32, 0, as_stream(stream)>>>(
        raw, nullptr, noise, noise_std, z, ray_norm, comp, weights, acc, depth, B, N, flags, 1e-10f, seed, offset, g_step_dev, idx0);
    NSB_LAUNCH_CHECK("composite_raw_fwd_kernel");
    return NSB_OK;
}
}  // namespace nsb

extern "C" int nsb_composite_raw_fwd(const float* raw, const float* noise, float noise_std, const float* z,
                                     const float* ray_norm, float* comp, float* weights, float* acc, float* depth,
                                     int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset, void* stream) {
    return composite_raw_fwd_at(raw, noise, noise_std, z, ray_norm, comp, weights, acc, depth, B, N, flags, seed, offset, 0, stream);
}

extern "C" int nsb_composite_raw_bwd_mse(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm,
                                         const float* target, float loss_scale, float* d_raw, int64_t B, int N, uint32_t flags,
                                         uint64_t seed, uint64_t offset, void* stream) {
    if (B == 0) return NSB_OK;
    if (!raw || !z || !target || !d_raw || N < 1 || B < 0) return NSB_E_BADARG;
    if (N <= kRunMaxN)
        return launch_bwd_run<true>(raw, nullptr, noise, noise_std, z, ray_norm, nullptr, nullptr, nullptr, nullptr, d_raw, nullptr, B, N, flags,
                                    1e-10f, seed, offset, stream, 0, target, loss_scale);
    return launch_bwd<true>(raw, nullptr, noise, noise_std, z, ray_norm, nullptr, nullptr, nullptr, nullptr, d_raw, nullptr, B, N, flags, 1e-10f,
                            seed, offset, stream, 0, target, loss_scale);
}

extern "C" int nsb_composite_raw_bwd_ex(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm,
                                        const float* g_comp, const float* g_weights, const float* g_acc, const float* g_depth, float* d_raw,
                                        int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset, void* stream) {
    if (B == 0) return NSB_OK;
    if (!raw || !z || !d_raw || N < 1 || B < 0 || (!g_comp && !g_weights && !g_acc && !g_depth)) return NSB_E_BADARG;
    if (N <= kRunMaxN)
        return launch_bwd_run<true>(raw, nullptr, noise, noise_std, z, ray_norm, g_comp, g_weights, g_acc, g_depth, d_raw, nullptr, B, N, flags,
                                    1e-10f, seed, offset, stream);
    return launch_bwd<true>(raw, nullptr, noise, noise_std, z, ray_norm, g_comp, g_weights, g_acc, g_depth, d_raw,
                            nullptr, B, N, flags, 1e-10f, seed, offset, stream);
}

extern "C" int nsb_composite_raw_bwd(const float* raw, const float* noise, float noise_std, const float* z,
                                     const float* ray_norm, const float* g_comp, float* d_raw, int64_t B, int N,
                                     uint32_t flags, uint64_t seed, uint64_t offset, void* stream) {
    if (B != 0 && !g_comp) return NSB_E_BADARG;
    return nsb_composite_raw_bwd_ex(raw, noise, noise_std, z, ray_norm, g_comp, nullptr, nullptr, nullptr, d_raw, B, N, flags, seed, offset,
                                    stream);
}

extern "C" int nsb_mse_loss(const float* comp_c, const float* comp_f, const float* target, float* g_c, float* g_f,
                            float* scalars, int64_t B, float grad_scale, void* stream) {
    if (!comp_f || !target || !scalars || B < 1) return NSB_E_BADARG;
    const int64_t n = B * 3;
    if (n <= 16384) {
        mse_single_block_kernel<<<1, 256, 0, as_stream(stream)>>>(comp_c, comp_f, target, g_c, g_f, scalars, n, grad_scale);
        NSB_LAUNCH_CHECK("mse_single_block_kernel");
        return NSB_OK;
    }
    mse_zero_kernel<<<1, 32, 0, as_stream(stream)>>>(scalars);
    NSB_LAUNCH_CHECK("mse_zero_kernel");
    const int grid = (int)(cdiv(n, 256) < 296 ? cdiv(n, 256) : 296);
    mse_loss_kernel<<<grid, 256, 0, as_stream(stream)>>>(comp_c, comp_f, target, g_c, g_f, scalars, n, grad_scale);
    NSB_LAUNCH_CHECK("mse_loss_kernel");
    mse_finish_kernel<<<1, 32, 0, as_stream(stream)>>>(scalars);
    NSB_LAUNCH_CHECK("mse_finish_kernel");
    return NSB_OK;
}
