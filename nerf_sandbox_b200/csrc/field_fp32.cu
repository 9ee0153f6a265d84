// K1 (fp32 mode) -- positional encoder + NeRF MLP with fp32 activations and gradients end to end.
// This is the 1e-4 parity mode of the field for training: one GEMM per layer and role on the tensor cores with bf16-split
// operands (field_split.cu) and the bias/ReLU/mask epilogues fused, concat-free activation layout
// (layer 3 writes straight into the [h | gamma(x)] buffer of the skip layer, `feature` into the
// [feat | gamma(d)] buffer of color_fc), dedicated warp-per-point kernels for the N=1/N=3 heads.
// The inference forward (no stash) and the bf16 mode live in field_tc.cu.
#include <cstdio>
#include <cstdlib>
#include "nsb_common.cuh"

namespace nsb {

// ---------------------------------------------------------------------------------------------------
// workspace carve-up (floats per point)
// ---------------------------------------------------------------------------------------------------
struct Fp32Ws {
    float *X0, *X4, *XC, *C;            // [Q,64] [Q,320] [Q,288] [Q,128]
    float* out[8];                      // output buffer of trunk layer l (ld = out_ld[l])
    int out_ld[8];
    float *dA, *dB, *dC;                // backward ping-pong [Q,256] x2, [Q,128]
    size_t bytes;
};

static Fp32Ws carve_fp32(void* base, int64_t Q) {
    Fp32Ws w;
    char* p = reinterpret_cast<char*>(base);
    size_t off = 0;
    auto take = [&](int64_t floats_per_pt) {
        float* r = reinterpret_cast<float*>(p + off);
        off += align_up((size_t)Q * floats_per_pt * sizeof(float), 256);
        return r;
    };
    w.X0 = take(kPosPad); w.X4 = take(kSkipPad); w.XC = take(kColorPad); w.C = take(kColorHidden);
    for (int l = 0; l < 8; ++l) {
        if (l == 3) { w.out[l] = w.X4; w.out_ld[l] = kSkipPad; }
        else { w.out[l] = take(kHidden); w.out_ld[l] = kHidden; }
    }
    w.dA = take(kHidden); w.dB = take(kHidden); w.dC = take(kColorHidden);
    w.bytes = off;
    return w;
}

// Without a stash (inference) the forward is field_tc.cu's fp16-split kernel, which uses no workspace.  The size reported
// for that case stays at the input buffers plus two hidden-layer buffers: nsb_field_workspace_bytes and
// nsb_render_workspace_bytes are part of the C ABI.
size_t fp32_workspace_bytes(int64_t Q, int stash) {
    if (stash) return carve_fp32(nullptr, Q).bytes;
    auto buf = [&](int64_t floats_per_pt) { return align_up((size_t)Q * floats_per_pt * sizeof(float), 256); };
    return buf(kPosPad) + buf(kSkipPad) + buf(kColorPad) + buf(kColorHidden) + 2 * buf(kHidden);
}

// ---------------------------------------------------------------------------------------------------
// encoders
// ---------------------------------------------------------------------------------------------------
// PositionalEncoder.forward, generic (models/encoders.py:88-106)
__global__ void encode_kernel(const float* __restrict__ x, float* __restrict__ out, int64_t Q, int D, int L,
                              int include_input) {
    const int od = D * (include_input ? 1 : 0) + 2 * L * D;
    const int64_t total = Q * od;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = idx / od;
        int j = (int)(idx % od);
        float v;
        if (include_input && j < D) v = x[q * D + j];
        else {
            j -= include_input ? D : 0;
            const bool is_cos = j >= L * D;
            if (is_cos) j -= L * D;
            const int k = j / D, d = j % D;
            const float arg = x[q * D + d] * exp2f((float)k);      // exact power-of-two scaling (:95)
            v = is_cos ? cosf(arg) : sinf(arg);
        }
        out[idx] = v;
    }
}

// PositionalEncoder backward: g_x[q,d] = [include] g[q,d] + sum_k 2^k (cos(2^k x) g_sin[k,d] - sin(2^k x) g_cos[k,d]), in the output
// order of encode_kernel; thread per (q, d).  sincosf is the accurate one, as in the forward: arguments reach 2^9 |x|.
__global__ void encode_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, float* __restrict__ gx, int64_t Q, int D, int L,
                                  int include_input) {
    const int od = D * (include_input ? 1 : 0) + 2 * L * D, o0 = include_input ? D : 0;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < Q * D; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = idx / D;
        const int d = (int)(idx % D);
        const float* gr = g + q * od;
        const float xv = x[idx];
        float acc = include_input ? gr[d] : 0.f;
        for (int k = 0; k < L; ++k) {
            const float f = exp2f((float)k);
            float sn, cs;
            sincosf(xv * f, &sn, &cs);
            acc += f * (cs * gr[o0 + k * D + d] - sn * gr[o0 + L * D + k * D + d]);
        }
        gx[idx] = acc;
    }
}

// Backward of the points + encodings step of nerf_forward_pass (render_utils.py:211-223) for gamma(x) (L = 10) and gamma(d)
// (L = 4), include_input, D = 3.  One warp per ray: lane i takes samples i, i + 32, ...; the sums over samples run in that fixed
// order and then through a fixed butterfly, so the input gradients are bitwise repeatable (no atomics).
//   pts = o + d * (z * norm)   ->  d_o = sum dx,  d_d = sum dx * (z * norm)
//   v = normalize(viewdirs or d, eps 1e-12)  ->  F.normalize backward of sum dv, into d_viewdirs (or d_d when viewdirs is null)
__global__ void __launch_bounds__(256)
encode_bwd_rays_kernel(const float* __restrict__ d_enc_pos, const float* __restrict__ d_enc_dir, const float* __restrict__ rays_o,
                       const float* __restrict__ rays_d, const float* __restrict__ z, const float* __restrict__ ray_norm,
                       const float* __restrict__ viewdirs, float* __restrict__ d_rays_o, float* __restrict__ d_rays_d,
                       float* __restrict__ d_viewdirs, int64_t B, int N) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = warp; b < B; b += nwarps) {
        const float o[3] = {rays_o[b * 3 + 0], rays_o[b * 3 + 1], rays_o[b * 3 + 2]};
        const float dd[3] = {rays_d[b * 3 + 0], rays_d[b * 3 + 1], rays_d[b * 3 + 2]};
        const float* vsrc = viewdirs ? viewdirs : rays_d;
        const float vr[3] = {vsrc[b * 3 + 0], vsrc[b * 3 + 1], vsrc[b * 3 + 2]};
        const float nv = sqrtf(vr[0] * vr[0] + vr[1] * vr[1] + vr[2] * vr[2]);
        const float nrm = fmaxf(nv, 1e-12f);
        const float v[3] = {vr[0] / nrm, vr[1] / nrm, vr[2] / nrm};
        float sx[3] = {0.f, 0.f, 0.f}, sxz[3] = {0.f, 0.f, 0.f}, sv[3] = {0.f, 0.f, 0.f};
        for (int i = lane; i < N; i += 32) {
            const int64_t q = b * N + i;
            const float zm = ray_norm ? __fmul_rn(z[q], ray_norm[b]) : z[q];
            const float* gp = d_enc_pos + q * kPosDim;
            const float* gd = d_enc_dir + q * kDirDim;
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const float p = __fadd_rn(o[d], __fmul_rn(dd[d], zm));
                float ax = gp[d];
#pragma unroll
                for (int k = 0; k < 10; ++k) {
                    const float f = exp2f((float)k);
                    float sn, cs;
                    sincosf(p * f, &sn, &cs);
                    ax += f * (cs * gp[3 + 3 * k + d] - sn * gp[33 + 3 * k + d]);
                }
                float av = gd[d];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float f = exp2f((float)k);
                    float sn, cs;
                    sincosf(v[d] * f, &sn, &cs);
                    av += f * (cs * gd[3 + 3 * k + d] - sn * gd[15 + 3 * k + d]);
                }
                sx[d] += ax; sxz[d] += ax * zm; sv[d] += av;
            }
        }
#pragma unroll
        for (int d = 0; d < 3; ++d) { sx[d] = warp_sum(sx[d]); sxz[d] = warp_sum(sxz[d]); sv[d] = warp_sum(sv[d]); }
        if (lane == 0) {
            // F.normalize: v = x / max(|x|, eps) -> dx = (g - v (v . g)) / |x| when |x| > eps, else g / eps
            float gvx[3];
            if (nv > 1e-12f) {
                const float vg = v[0] * sv[0] + v[1] * sv[1] + v[2] * sv[2];
#pragma unroll
                for (int d = 0; d < 3; ++d) gvx[d] = (sv[d] - v[d] * vg) / nv;
            } else {
#pragma unroll
                for (int d = 0; d < 3; ++d) gvx[d] = sv[d] / 1e-12f;
            }
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                if (d_rays_o) d_rays_o[b * 3 + d] = sx[d];
                if (d_rays_d) d_rays_d[b * 3 + d] = sxz[d] + (viewdirs ? 0.f : gvx[d]);
                if (d_viewdirs && viewdirs) d_viewdirs[b * 3 + d] = gvx[d];
            }
        }
    }
}

// points + both encodings into the padded activation buffers; 16 threads per point
__global__ void prepare_from_rays_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                         const float* __restrict__ z, const float* __restrict__ ray_norm,
                                         const float* __restrict__ viewdirs, float* __restrict__ X0,
                                         float* __restrict__ X4, float* __restrict__ XC, int64_t B, int N) {
    const int64_t Q = B * (int64_t)N;
    const int sub = threadIdx.x & 15;
    for (int64_t q = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 4; q < Q;
         q += ((int64_t)gridDim.x * blockDim.x) >> 4) {
        const int64_t b = q / N;
        if (sub < 10 || sub == 14) {
            // render_utils.py:211-215 -- z*norm, then d*that, then + o, each rounded separately
            const float zm = ray_norm ? __fmul_rn(z[q], ray_norm[b]) : z[q];
            float p[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) p[d] = __fadd_rn(rays_o[b * 3 + d], __fmul_rn(rays_d[b * 3 + d], zm));
            float* r0 = X0 + q * kPosPad;
            float* r4 = X4 + q * kSkipPad + kHidden;
            if (sub == 14) {
#pragma unroll
                for (int d = 0; d < 3; ++d) { r0[d] = p[d]; r4[d] = p[d]; }
                r0[63] = 0.f; r4[63] = 0.f;
            } else {
                const float f = exp2f((float)sub);
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    float s, c;
                    sincosf(p[d] * f, &s, &c);
                    r0[3 + 3 * sub + d] = s; r0[33 + 3 * sub + d] = c;
                    r4[3 + 3 * sub + d] = s; r4[33 + 3 * sub + d] = c;
                }
            }
        } else {
            const float* vsrc = viewdirs ? viewdirs : rays_d;        // :218-222
            const float vx = vsrc[b * 3 + 0], vy = vsrc[b * 3 + 1], vz = vsrc[b * 3 + 2];
            const float nrm = fmaxf(sqrtf(vx * vx + vy * vy + vz * vz), 1e-12f);   // F.normalize
            const float v[3] = {vx / nrm, vy / nrm, vz / nrm};
            float* rc = XC + q * kColorPad + kHidden;
            if (sub == 15) {
#pragma unroll
                for (int d = 0; d < 3; ++d) rc[d] = v[d];
                for (int j = kDirDim; j < kColorPad - kHidden; ++j) rc[j] = 0.f;
            } else {
                const int k = sub - 10;
                const float f = exp2f((float)k);
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    float s, c;
                    sincosf(v[d] * f, &s, &c);
                    rc[3 + 3 * k + d] = s; rc[15 + 3 * k + d] = c;
                }
            }
        }
    }
}

// materialised encodings -> padded buffers (NeRF.forward module boundary)
__global__ void prepare_from_enc_kernel(const float* __restrict__ enc_pos, const float* __restrict__ enc_dir,
                                        float* __restrict__ X0, float* __restrict__ X4, float* __restrict__ XC,
                                        int64_t Q) {
    const int64_t total = Q * 96;       // 64 pos slots + 32 dir slots per point
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = idx / 96;
        const int j = (int)(idx % 96);
        if (j < 64) {
            const float v = j < kPosDim ? enc_pos[q * kPosDim + j] : 0.f;
            X0[q * kPosPad + j] = v; X4[q * kSkipPad + kHidden + j] = v;
        } else {
            const int jj = j - 64;
            XC[q * kColorPad + kHidden + jj] = jj < kDirDim ? enc_dir[q * kDirDim + jj] : 0.f;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// heads: sigma_out (256->1) and color_out (128->3), warp per point
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
head_fwd_kernel(const float* __restrict__ C, const float* __restrict__ H8, int64_t ldh, const float* __restrict__ Wo,
                const float* __restrict__ bo, const float* __restrict__ ws, const float* __restrict__ bs,
                float* __restrict__ raw, int64_t Q) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(Wo) + lane);
    const float4 w1 = __ldg(reinterpret_cast<const float4*>(Wo + 128) + lane);
    const float4 w2 = __ldg(reinterpret_cast<const float4*>(Wo + 256) + lane);
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(ws) + lane);
    const float4 s1 = __ldg(reinterpret_cast<const float4*>(ws) + 32 + lane);
    for (int64_t q = warp; q < Q; q += nwarps) {
        const float4 c = *(reinterpret_cast<const float4*>(C + q * kColorHidden) + lane);
        const float4 h0 = *(reinterpret_cast<const float4*>(H8 + q * ldh) + lane);
        const float4 h1 = *(reinterpret_cast<const float4*>(H8 + q * ldh) + 32 + lane);
        float r = c.x * w0.x + c.y * w0.y + c.z * w0.z + c.w * w0.w;
        float g = c.x * w1.x + c.y * w1.y + c.z * w1.z + c.w * w1.w;
        float b = c.x * w2.x + c.y * w2.y + c.z * w2.z + c.w * w2.w;
        float s = h0.x * s0.x + h0.y * s0.y + h0.z * s0.z + h0.w * s0.w + h1.x * s1.x + h1.y * s1.y + h1.z * s1.z + h1.w * s1.w;
        r = warp_sum(r); g = warp_sum(g); b = warp_sum(b); s = warp_sum(s);
        if (lane == 0) reinterpret_cast<float4*>(raw)[q] = make_float4(r + bo[0], g + bo[1], b + bo[2], s + bs[0]);
    }
}

// d_raw -> dC (masked by c>0), dH8 seed (= d_sigma * w_sigma), and the head parameter grads
__global__ void __launch_bounds__(256)
head_bwd_kernel(const float* __restrict__ d_raw, const float* __restrict__ C, const float* __restrict__ H8, int64_t ldh,
                const float* __restrict__ Wo, const float* __restrict__ ws, float* __restrict__ dC,
                float* __restrict__ dH8, float* __restrict__ gWo, float* __restrict__ gbo, float* __restrict__ gws,
                float* __restrict__ gbs, int64_t Q) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(Wo) + lane);
    const float4 w1 = __ldg(reinterpret_cast<const float4*>(Wo + 128) + lane);
    const float4 w2 = __ldg(reinterpret_cast<const float4*>(Wo + 256) + lane);
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(ws) + lane);
    const float4 s1 = __ldg(reinterpret_cast<const float4*>(ws) + 32 + lane);
    float4 a0 = make_float4(0, 0, 0, 0), a1 = a0, a2 = a0, as0 = a0, as1 = a0;
    float b0 = 0.f, b1 = 0.f, b2 = 0.f, bsig = 0.f;
    for (int64_t q = warp; q < Q; q += nwarps) {
        const float4 d = __ldg(reinterpret_cast<const float4*>(d_raw) + q);
        const float4 c = *(reinterpret_cast<const float4*>(C + q * kColorHidden) + lane);
        const float4 h0 = *(reinterpret_cast<const float4*>(H8 + q * ldh) + lane);
        const float4 h1 = *(reinterpret_cast<const float4*>(H8 + q * ldh) + 32 + lane);
        float4 dc;
        dc.x = c.x > 0.f ? d.x * w0.x + d.y * w1.x + d.z * w2.x : 0.f;
        dc.y = c.y > 0.f ? d.x * w0.y + d.y * w1.y + d.z * w2.y : 0.f;
        dc.z = c.z > 0.f ? d.x * w0.z + d.y * w1.z + d.z * w2.z : 0.f;
        dc.w = c.w > 0.f ? d.x * w0.w + d.y * w1.w + d.z * w2.w : 0.f;
        *(reinterpret_cast<float4*>(dC + q * kColorHidden) + lane) = dc;
        *(reinterpret_cast<float4*>(dH8 + q * kHidden) + lane) = make_float4(d.w * s0.x, d.w * s0.y, d.w * s0.z, d.w * s0.w);
        *(reinterpret_cast<float4*>(dH8 + q * kHidden) + 32 + lane) = make_float4(d.w * s1.x, d.w * s1.y, d.w * s1.z, d.w * s1.w);
        a0.x += d.x * c.x; a0.y += d.x * c.y; a0.z += d.x * c.z; a0.w += d.x * c.w;
        a1.x += d.y * c.x; a1.y += d.y * c.y; a1.z += d.y * c.z; a1.w += d.y * c.w;
        a2.x += d.z * c.x; a2.y += d.z * c.y; a2.z += d.z * c.z; a2.w += d.z * c.w;
        as0.x += d.w * h0.x; as0.y += d.w * h0.y; as0.z += d.w * h0.z; as0.w += d.w * h0.w;
        as1.x += d.w * h1.x; as1.y += d.w * h1.y; as1.z += d.w * h1.z; as1.w += d.w * h1.w;
        if (lane == 0) { b0 += d.x; b1 += d.y; b2 += d.z; bsig += d.w; }
    }
    if (gWo == nullptr) return;          // frozen field: input gradients only
    // block-level reduction in shared memory, then one atomic per element per block
    __shared__ float red[3 * 128 + 256 + 4];
    for (int i = threadIdx.x; i < 3 * 128 + 256 + 4; i += blockDim.x) red[i] = 0.f;
    __syncthreads();
    const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w}, av2[4] = {a2.x, a2.y, a2.z, a2.w};
    const float sv0[4] = {as0.x, as0.y, as0.z, as0.w}, sv1[4] = {as1.x, as1.y, as1.z, as1.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        atomicAdd(&red[lane * 4 + j], av0[j]); atomicAdd(&red[128 + lane * 4 + j], av1[j]);
        atomicAdd(&red[256 + lane * 4 + j], av2[j]);
        atomicAdd(&red[384 + lane * 4 + j], sv0[j]); atomicAdd(&red[384 + 128 + lane * 4 + j], sv1[j]);
    }
    if (lane == 0) { atomicAdd(&red[640], b0); atomicAdd(&red[641], b1); atomicAdd(&red[642], b2); atomicAdd(&red[643], bsig); }
    __syncthreads();
    for (int i = threadIdx.x; i < 644; i += blockDim.x) {
        const float v = red[i];
        if (i < 384) atomicAdd(gWo + i, v);
        else if (i < 640) atomicAdd(gws + (i - 384), v);
        else if (i < 643) atomicAdd(gbo + (i - 640), v);
        else atomicAdd(gbs, v);
    }
}

// ---------------------------------------------------------------------------------------------------
// weight packing (fp32 section): flat state_dict order -> rows padded to Kpad, zero filled
// ---------------------------------------------------------------------------------------------------
struct PackFp32Args { size_t w[12], b[12]; };
__global__ void pack_fp32_kernel(const float* __restrict__ params, char* __restrict__ base, PackFp32Args a) {
    const int l = blockIdx.y;
    const LayerDesc d = layer_desc(l);
    float* dstw = reinterpret_cast<float*>(base + a.w[l]);
    float* dstb = reinterpret_cast<float*>(base + a.b[l]);
    const int total = d.N * d.Kpad;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int n = idx / d.Kpad, k = idx % d.Kpad;
        dstw[idx] = k < d.K ? params[d.w_off + (int64_t)n * d.K + k] : 0.f;
    }
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < d.N; n += gridDim.x * blockDim.x) dstb[n] = params[d.b_off + n];
}

PackedLayout packed_layout() {
    PackedLayout L;
    size_t off = 0;
    for (int l = 0; l < 12; ++l) {
        const LayerDesc d = layer_desc(l);
        L.f32_w[l] = off; off += align_up((size_t)d.N * d.Kpad * sizeof(float), 256);
        L.f32_b[l] = off; off += align_up((size_t)d.N * sizeof(float), 256);
    }
    L.bf16_off = off;
    L.bf16_bytes = tc_packed_bytes();
    off += L.bf16_bytes;
    L.split_off = off;
    for (int l = 0; l < 12; ++l) {
        const LayerDesc d = layer_desc(l);
        L.split_fwd[l] = L.split_dgrad[l] = 0;
        if (l == 9 || l == 11) continue;                       // sigma_out / color_out are CUDA-core heads
        L.split_fwd[l] = off; off += align_up(split_image_bytes(d.N, d.Kpad), 256);
        if (l > 0) { L.split_dgrad[l] = off; off += align_up(split_image_bytes(kHidden, d.N), 256); }
    }
    for (int i = 0; i < 3; ++i) {                              // W_0[:, 0:63]^T, W_4[:, 256:319]^T (64 rows), W_cfc[:, 256:283]^T (32)
        L.split_dinput[i] = off;
        off += align_up(split_image_bytes(i < 2 ? 64 : 32, i < 2 ? kHidden : kColorHidden), 256);
    }
    L.split_bytes = off - L.split_off;
    L.total = off;
    return L;
}

int pack_fp32(const float* params, void* packed, cudaStream_t st) {
    const PackedLayout L = packed_layout();
    PackFp32Args a;
    for (int l = 0; l < 12; ++l) { a.w[l] = L.f32_w[l]; a.b[l] = L.f32_b[l]; }
    pack_fp32_kernel<<<dim3(32, 12), 256, 0, st>>>(params, reinterpret_cast<char*>(packed), a);
    NSB_LAUNCH_CHECK("pack_fp32_kernel");
    return split_pack(params, packed, st);
}

// ---------------------------------------------------------------------------------------------------
// host orchestration
// ---------------------------------------------------------------------------------------------------
static inline const float* PW(const void* packed, const PackedLayout& L, int l) {
    return reinterpret_cast<const float*>(reinterpret_cast<const char*>(packed) + L.f32_w[l]);
}
static inline const float* PB(const void* packed, const PackedLayout& L, int l) {
    return reinterpret_cast<const float*>(reinterpret_cast<const char*>(packed) + L.f32_b[l]);
}
static inline const uint8_t* IMG(const void* packed, size_t off) { return reinterpret_cast<const uint8_t*>(packed) + off; }

// The layer GEMMs run on the tensor cores with bf16-split operands (field_split.cu).  The forward, dgrad and input-gradient
// GEMMs take the weights (their B operand) from the term images split_pack writes into the packed weights.
static int gemm_fwd(const float* X, int64_t ldx, const uint8_t* w_img, int Kpad, const float* bias, float* Y, int64_t ldy,
                    int64_t Q, int N, int relu, cudaStream_t st) {
    GemmArgs g{};
    g.A = X; g.lda = ldx; g.C = Y; g.ldc = ldy; g.Mdim = Q; g.Ndim = N; g.Kdim = Kpad;
    g.bias = bias; g.relu = relu; g.b_img = w_img;
    return split_gemm(g, EPI_FWD, st);
}
// dX[Q, n_in] = dY[Q, n_out] . W[n_out, :n_in], (+addend) (*mask)
static int gemm_dgrad(const float* dY, int64_t ldy, const uint8_t* w_img, float* dX, int64_t ldx, int64_t Q, int n_out, int n_in,
                      const float* mask, int64_t ldm, const float* addend, int64_t ldadd, cudaStream_t st) {
    GemmArgs g{};
    g.A = dY; g.lda = ldy; g.C = dX; g.ldc = ldx; g.Mdim = Q; g.Ndim = n_in; g.Kdim = n_out;
    g.mask = mask; g.ldm = ldm; g.addend = addend; g.ldadd = ldadd; g.b_img = w_img;
    return split_gemm(g, EPI_DGRAD, st);
}
// Input gradient: dE[Q, n_valid] (row stride lde, any) = dY[Q, n_out] . W_slice[n_out, n_in] (n_in a multiple of 16 covering
// n_valid; the image's padding columns are zero) (+ addend, same layout as dE)
static int gemm_dinput(const float* dY, int64_t ldy, const uint8_t* w_img, float* dE, int64_t lde, int64_t Q, int n_out, int n_in,
                       int n_valid, const float* addend, cudaStream_t st) {
    GemmArgs g{};
    g.A = dY; g.lda = ldy; g.C = dE; g.ldc = lde; g.Mdim = Q; g.Ndim = n_in; g.Kdim = n_out;
    g.addend = addend; g.ldadd = lde; g.n_valid = n_valid; g.b_img = w_img;
    return split_gemm(g, EPI_DGRAD, st);
}
// gW[n_out, K] += dY[Q, n_out]^T . X[Q, Kpad] ; gb[n_out] += colsum(dY)
static int gemm_wgrad(const float* dY, int64_t ldy, const float* X, int64_t ldx, float* gW, float* gb, int64_t Q,
                      int n_out, int K, int Kpad, cudaStream_t st) {
    GemmArgs g{};
    g.A = dY; g.lda = ldy; g.B = X; g.ldb = ldx; g.C = gW; g.ldc = K; g.Mdim = n_out; g.Ndim = Kpad; g.Kdim = Q;
    g.n_valid = K;
    g.colsum = gb;                      // the bias gradient rides along (the kernel sees every dY element anyway)
    return split_gemm(g, EPI_WGRAD, st);
}

static int elem_grid(int64_t total) {
    const int64_t want = cdiv(total, 256), cap = (int64_t)num_sms() * 16;
    return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

int fp32_prepare_rays(const float* o, const float* d, const float* z, const float* rn, const float* vd, void* ws,
                      int64_t B, int N, cudaStream_t st) {
    Fp32Ws w = carve_fp32(ws, B * (int64_t)N);
    prepare_from_rays_kernel<<<elem_grid(B * (int64_t)N * 16), 256, 0, st>>>(o, d, z, rn, vd, w.X0, w.X4, w.XC, B, N);
    NSB_LAUNCH_CHECK("prepare_from_rays_kernel");
    return NSB_OK;
}
int fp32_prepare_enc(const float* ep, const float* ed, void* ws, int64_t Q, cudaStream_t st) {
    Fp32Ws w = carve_fp32(ws, Q);
    prepare_from_enc_kernel<<<elem_grid(Q * 96), 256, 0, st>>>(ep, ed, w.X0, w.X4, w.XC, Q);
    NSB_LAUNCH_CHECK("prepare_from_enc_kernel");
    return NSB_OK;
}

// mlps.py:221-278 on the prepared buffers
int fp32_mlp_fwd(const void* packed, float* raw, void* ws, int64_t Q, cudaStream_t st) {
    const PackedLayout L = packed_layout();
    Fp32Ws w = carve_fp32(ws, Q);
    const float* in = w.X0; int64_t ldin = kPosPad;
    for (int l = 0; l < 8; ++l) {
        const LayerDesc d = layer_desc(l);
        if (l == 4) { in = w.X4; ldin = kSkipPad; }
        NSB_TRY(gemm_fwd(in, ldin, IMG(packed, L.split_fwd[l]), d.Kpad, PB(packed, L, l), w.out[l], w.out_ld[l], Q, 256, 1, st));
        in = w.out[l]; ldin = w.out_ld[l];
    }
    const float* H8 = w.out[7];
    NSB_TRY(gemm_fwd(H8, kHidden, IMG(packed, L.split_fwd[8]), 256, PB(packed, L, 8), w.XC, kColorPad, Q, 256, 0, st));       // feature
    NSB_TRY(gemm_fwd(w.XC, kColorPad, IMG(packed, L.split_fwd[10]), kColorPad, PB(packed, L, 10), w.C, kColorHidden, Q, 128, 1, st));  // color_fc
    head_fwd_kernel<<<elem_grid(Q * 32), 256, 0, st>>>(w.C, H8, kHidden, PW(packed, L, 11), PB(packed, L, 11),
                                                      PW(packed, L, 9), PB(packed, L, 9), raw, Q);
    NSB_LAUNCH_CHECK("head_fwd_kernel");
    return NSB_OK;
}

// Parameter grads (accumulated into flat `grads`, or none when it is null: a frozen field) and the gradients w.r.t. the two
// encodings (d_enc_pos [Q,63], d_enc_dir [Q,27], each optional) from the stashed activations:
//   d gamma(d) = dY_9 . W_cfc[:, 256:283],   d gamma(x) = dY_0 . W_0 + dY_4 . W_4[:, 256:319]   (layer 4's input is [h | gamma(x)])
int fp32_mlp_bwd(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws, int64_t Q,
                 cudaStream_t st) {
    const PackedLayout L = packed_layout();
    Fp32Ws w = carve_fp32(ws, Q);
    const float* H8 = w.out[7];
    const LayerDesc dsg = layer_desc(9), dco = layer_desc(11), dfc = layer_desc(10), dft = layer_desc(8);
    auto G = [&](int64_t off) { return grads ? grads + off : nullptr; };
    int hb_grid = num_sms() * 4;
    if ((int64_t)hb_grid * 8 > Q) hb_grid = (int)cdiv(Q, 8);
    head_bwd_kernel<<<hb_grid, 256, 0, st>>>(d_raw, w.C, H8, kHidden, PW(packed, L, 11), PW(packed, L, 9), w.dC, w.dA,
                                             G(dco.w_off), G(dco.b_off), G(dsg.w_off), G(dsg.b_off), Q);
    NSB_LAUNCH_CHECK("head_bwd_kernel");
    if (d_enc_dir)
        NSB_TRY(gemm_dinput(w.dC, kColorHidden, IMG(packed, L.split_dinput[2]), d_enc_dir, kDirDim, Q, kColorHidden, 32, kDirDim, nullptr, st));
    if (!grads && !d_enc_pos) return NSB_OK;
    // color_fc
    if (grads) NSB_TRY(gemm_wgrad(w.dC, kColorHidden, w.XC, kColorPad, grads + dfc.w_off, grads + dfc.b_off, Q, 128, dfc.K, dfc.Kpad, st));
    NSB_TRY(gemm_dgrad(w.dC, kColorHidden, IMG(packed, L.split_dgrad[10]), w.dB, kHidden, Q, 128, 256, nullptr, 0, nullptr, 0, st));  // dFeat
    // feature (no activation); dH8 = (dFeat.Wf + dsigma*w_sigma) * (H8>0)
    if (grads) NSB_TRY(gemm_wgrad(w.dB, kHidden, H8, kHidden, grads + dft.w_off, grads + dft.b_off, Q, 256, 256, 256, st));
    NSB_TRY(gemm_dgrad(w.dB, kHidden, IMG(packed, L.split_dgrad[8]), w.dA, kHidden, Q, 256, 256, H8, kHidden, w.dA, kHidden, st));
    float* dcur = w.dA; float* dnext = w.dB;
    for (int l = 7; l >= 0; --l) {
        const LayerDesc d = layer_desc(l);
        const float* Xin = l == 0 ? w.X0 : (l == 4 ? w.X4 : w.out[l - 1]);
        const int64_t ldx = l == 0 ? kPosPad : (l == 4 ? kSkipPad : w.out_ld[l - 1]);
        if (grads) NSB_TRY(gemm_wgrad(dcur, kHidden, Xin, ldx, grads + d.w_off, grads + d.b_off, Q, 256, d.K, d.Kpad, st));
        if (d_enc_pos && l == 4)        // the gamma(x) slab of the skip input, before the ping-pong overwrites dY_4
            NSB_TRY(gemm_dinput(dcur, kHidden, IMG(packed, L.split_dinput[1]), d_enc_pos, kPosDim, Q, kHidden, kPosPad, kPosDim, nullptr, st));
        if (d_enc_pos && l == 0)
            NSB_TRY(gemm_dinput(dcur, kHidden, IMG(packed, L.split_dinput[0]), d_enc_pos, kPosDim, Q, kHidden, kPosPad, kPosDim, d_enc_pos, st));
        if (l > 0) {
            // input of layer l is relu(out[l-1]) -> mask by out[l-1] > 0 (first 256 columns only at the skip layer)
            NSB_TRY(gemm_dgrad(dcur, kHidden, IMG(packed, L.split_dgrad[l]), dnext, kHidden, Q, 256, 256, w.out[l - 1], w.out_ld[l - 1],
                               nullptr, 0, st));
            float* t = dcur; dcur = dnext; dnext = t;
        }
    }
    return NSB_OK;
}

// ---- Adam --------------------------------------------------------------------------------------------
// bias corrections of step t = *t_dev + 1 (CUDA-graph replay: the step count lives in device memory); with T_max > 0 the
// learning rate follows CosineAnnealingLR(T_max, eta_min) after *t_dev scheduler steps (make_scheduler, train/trainer.py:81-88)
__device__ __forceinline__ void adam_bias_corrections(const uint64_t* t_dev, float lr, float eta_min, int64_t T_max, float b1, float b2,
                                                      float& lr_over_bc1, float& inv_sqrt_bc2) {
    __shared__ float s_bc[2];
    if (threadIdx.x == 0) {
        const double t = (double)(*t_dev + 1);
        if (T_max > 0) lr = (float)((double)eta_min + ((double)lr - (double)eta_min) * (1.0 + cos(3.141592653589793 * (double)*t_dev / (double)T_max)) * 0.5);
        s_bc[0] = (float)((double)lr / (1.0 - pow((double)b1, t)));
        s_bc[1] = (float)(1.0 / sqrt(1.0 - pow((double)b2, t)));
    }
    __syncthreads();
    lr_over_bc1 = s_bc[0]; inv_sqrt_bc2 = s_bc[1];
}
// One Adam element update with every rounding spelled out (no compiler-chosen FMA contraction): the plain kernel and the
// fused all-reduce kernel must produce bit-identical parameters from the same gradient (tests/test_gpu_dist.py).
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, float grad_scale, float b1, float b2, float eps,
                                            float lr_over_bc1, float inv_sqrt_bc2) {
    const float gi = __fmul_rn(g, grad_scale);
    m = __fmaf_rn(b1, m, __fmul_rn(1.0f - b1, gi));
    v = __fmaf_rn(b2, v, __fmul_rn(__fmul_rn(1.0f - b2, gi), gi));
    p = __fsub_rn(p, __fmul_rn(lr_over_bc1, __fdiv_rn(m, __fmaf_rn(__fsqrt_rn(v), inv_sqrt_bc2, eps))));
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr_over_bc1, float b1, float b2, float eps,
                            float inv_sqrt_bc2, float grad_scale, const uint64_t* t_dev, float lr, float eta_min, int64_t T_max,
                            const float* __restrict__ loss_guard) {
    // non-finite loss: the reference skips the optimiser step (train/trainer.py:713-716)
    if (loss_guard && !isfinite(*loss_guard)) return;
    if (t_dev) adam_bias_corrections(t_dev, lr, eta_min, T_max, b1, b2, lr_over_bc1, inv_sqrt_bc2);
    // 16-byte accesses when the buffers allow it (the flat parameter buffers do: 595,844 = 4 x 148,961)
    const bool vec = (n & 3) == 0 && ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                                       reinterpret_cast<uintptr_t>(v)) & 15) == 0;
    if (vec) {
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (n >> 2); i += (int64_t)gridDim.x * blockDim.x) {
            const float4 g4 = reinterpret_cast<const float4*>(g)[i];
            float4 m4 = reinterpret_cast<float4*>(m)[i], v4 = reinterpret_cast<float4*>(v)[i], p4 = reinterpret_cast<float4*>(p)[i];
            const float* gg = &g4.x; float* mm = &m4.x; float* vv = &v4.x; float* pp = &p4.x;
#pragma unroll
            for (int c = 0; c < 4; ++c) adam_update(pp[c], mm[c], vv[c], gg[c], grad_scale, b1, b2, eps, lr_over_bc1, inv_sqrt_bc2);
            reinterpret_cast<float4*>(m)[i] = m4; reinterpret_cast<float4*>(v)[i] = v4; reinterpret_cast<float4*>(p)[i] = p4;
        }
        return;
    }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float pi = p[i], mi = m[i], vi = v[i];
        adam_update(pi, mi, vi, g[i], grad_scale, b1, b2, eps, lr_over_bc1, inv_sqrt_bc2);
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
}

// ---- data-parallel step tail: all-reduce of the gradient buffers through peer memory + Adam, one kernel ----------------
// Every rank sums the `world` gradient buffers itself, in rank order (so the replicas stay bit-identical), with loads that
// go straight to the peers' HBM over NVLink / NVSwitch, and applies Adam to its full parameter copy.  The only
// synchronisation is a flag exchange at the top of the kernel: block 0 publishes "my gradients of this epoch are complete"
// into every peer's flag block (release, system scope), every block waits until its own flag block shows the epoch for all
// ranks (acquire).  The caller double-buffers the gradients (epoch parity), so no second barrier is needed: a rank can
// only overwrite a buffer two epochs later, after every peer has announced the epoch in between.
constexpr int kMaxPeers = 16;
constexpr int kMaxNets = 4;
struct AdamArParams {
    float* p[kMaxNets]; float* m[kMaxNets]; float* v[kMaxNets];   // n floats each; net k's gradients are grads[r] + k * n
    const float* grads[kMaxPeers];          // every rank's gradient buffer (peer-mapped addresses), n_nets * n floats
    const float* mc_grads;                  // multicast address of the same buffers (NVLS), or null
    float* mc_red;                          // two-phase NVLS exchange: multicast address of the REDUCED-gradient buffers, or null
    const float* red;                       // ... this rank's reduced-gradient buffer (n_nets * n floats)
    int* local_sync;                        // ... device ints of this rank: [0] finished-block counter, [1] epoch whose update is
                                            //     skipped, [2] epoch in which a peer timed out (4 ints, zeroed once)
    uint32_t* flags[kMaxPeers];             // every rank's flag block, uint32[world]
    int rank, world, n_nets; uint32_t epoch;
    int64_t n; float lr_over_bc1, b1, b2, eps, inv_sqrt_bc2, grad_scale;
    const uint64_t* t_dev; float lr, eta_min; int64_t T_max;       // graph replay: step count (and epoch) = *t_dev + 1
    const float* loss_guard;                // this rank's loss (device), or null: a non-finite loss on ANY rank skips the update
    uint64_t timeout_ns;                    // how long a rank waits for its peers' flags before it gives up (NSB_PEER_TIMEOUT_S)
};
// Set (1 + peer rank) by a rank that gave up waiting for `peer`; read by the host through nsb_peer_status().  A rank that
// times out leaves the kernel WITHOUT applying the update and without killing the context -- the host raises.
__device__ unsigned int g_peer_error = 0;
__device__ __forceinline__ uint64_t ar_global_ns() { uint64_t t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
// NVLS: one load returns the sum over every rank's copy, reduced inside the NVSwitch
__device__ __forceinline__ float4 ld_reduce_mc(const float4* p) {
    float4 x;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                 : "l"(p) : "memory");
    return x;
}
__device__ __forceinline__ float4 ld_peer(const float4* p) {
    float4 x;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "l"(p));
    return x;
}
template <int WORLD>      // 0: run-time world size
__global__ void __launch_bounds__(256) adam_allreduce_kernel(const __grid_constant__ AdamArParams a) {
    const int world = WORLD ? WORLD : a.world;
    float lr_over_bc1 = a.lr_over_bc1, inv_sqrt_bc2 = a.inv_sqrt_bc2;
    uint32_t epoch = a.epoch;
    if (a.t_dev) { adam_bias_corrections(a.t_dev, a.lr, a.eta_min, a.T_max, a.b1, a.b2, lr_over_bc1, inv_sqrt_bc2); epoch = (uint32_t)(*a.t_dev + 1); }
    __shared__ int s_abort;
    // train/trainer.py:713-716: a non-finite loss skips the optimiser step.  Across ranks the decision must be common, so
    // every rank publishes "my loss is bad" next to its epoch flag (one word per rank and epoch parity) and skips if any is.
    const uint32_t bad = (a.loss_guard && !isfinite(*a.loss_guard)) ? 1u : 0u;
    if (threadIdx.x == 0) s_abort = (world == 1 && bad) ? 1 : 0;
    __syncthreads();
    if (world > 1 && threadIdx.x < world) {     // (a single rank has nobody to wait for)
        const int r = threadIdx.x;
        const int bad_ofs = world * (1 + (int)(epoch & 1u));
        if (blockIdx.x == 0) {      // the gradient kernels of this stream have finished: publish that to rank r
            asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(a.flags[r] + bad_ofs + a.rank), "r"(bad) : "memory");
            __threadfence_system();
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flags[r] + a.rank), "r"(epoch) : "memory");
        }
        uint32_t seen;
        uint64_t t0 = 0;
        for (uint32_t i = 1;; ++i) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.flags[a.rank] + r) : "memory");
            if ((int32_t)(seen - epoch) >= 0) break;
            if (i & 0x3FFu) continue;
            if (t0 == 0) { t0 = ar_global_ns(); continue; }
            if (ar_global_ns() - t0 > a.timeout_ns) {
                // a peer never arrived (default: 10 min of skew -- validation, checkpointing or a data stall on one rank are
                // ordinary): record who, skip the update, let the host raise.  No __trap: the context stays usable.
                if (blockIdx.x == 0) printf("nsb adam_allreduce: rank %d gave up waiting for rank %d at epoch %u\n", a.rank, r, epoch);
                atomicMax(&g_peer_error, 1u + (unsigned)r);
                s_abort = 1;
                break;
            }
        }
        uint32_t peer_bad;
        asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(peer_bad) : "l"(a.flags[a.rank] + bad_ofs + r) : "memory");
        if (peer_bad) s_abort = 1;
    }
    __syncthreads();
    if (s_abort) return;
    const int64_t n4 = a.n >> 2, total4 = n4 * a.n_nets;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / n4);
        const int64_t j = i - k * n4;
        // all peers' loads in flight before the first add; summed in rank order: identical on every rank
        float4 x[WORLD ? WORLD : 1];
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.mc_grads) {
            g = ld_reduce_mc(reinterpret_cast<const float4*>(a.mc_grads) + i);
        } else if (WORLD) {
#pragma unroll
            for (int r = 0; r < (WORLD ? WORLD : 1); ++r) x[r] = ld_peer(reinterpret_cast<const float4*>(a.grads[r]) + i);
#pragma unroll
            for (int r = 0; r < (WORLD ? WORLD : 1); ++r) { g.x += x[r].x; g.y += x[r].y; g.z += x[r].z; g.w += x[r].w; }
        } else {
            for (int r = 0; r < world; ++r) {
                const float4 y = ld_peer(reinterpret_cast<const float4*>(a.grads[r]) + i);
                g.x += y.x; g.y += y.y; g.z += y.z; g.w += y.w;
            }
        }
        float4 pm = reinterpret_cast<float4*>(a.m[k])[j], pv = reinterpret_cast<float4*>(a.v[k])[j], pp = reinterpret_cast<float4*>(a.p[k])[j];
        float* gg = &g.x; float* mm = &pm.x; float* vv = &pv.x; float* pq = &pp.x;
#pragma unroll
        for (int c = 0; c < 4; ++c) adam_update(pq[c], mm[c], vv[c], gg[c], a.grad_scale, a.b1, a.b2, a.eps, lr_over_bc1, inv_sqrt_bc2);
        reinterpret_cast<float4*>(a.m[k])[j] = pm; reinterpret_cast<float4*>(a.v[k])[j] = pv; reinterpret_cast<float4*>(a.p[k])[j] = pp;
    }
}

// ---- two-phase exchange through the NVSwitch (4+ ranks) ------------------------------------------------------------------
// In the one-kernel exchange above EVERY rank pulls the WHOLE reduced buffer through `multimem.ld_reduce`: the switch then
// reads each GPU's 4.77 MB once per requester, i.e. 8 x 4.77 MB leave every GPU at 8 ranks (~55 us at NVLink rate; the same
// volume as reading seven peers' buffers, which is why NVLS barely beat the peer loads in round 1).  Bandwidth-optimal is
// reduce-scatter + all-gather: rank r reduces only ITS 1/world slice (its GPU sends and receives 4.77 MB in total) and
// multicast-STORES the result into every rank's `red` buffer (`multimem.st`); a second flag round, then every rank runs Adam
// on its local copy.  Two kernels, so no block ever waits on another block of its own grid: kernel 1's blocks wait only for
// the peers' "gradients complete" flags, kernel 2 (stream-ordered after kernel 1) only for the peers' "slice stored" flags.
__device__ __forceinline__ void st_mc(float4* p, const float4& x) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w) : "memory");
}
// wait until every rank's word at flags[own][base + r] has reached `epoch`; returns false on timeout (recorded in g_peer_error)
__device__ __forceinline__ bool wait_peer_flags(const AdamArParams& a, int base, int r, uint32_t epoch) {
    uint32_t seen;
    uint64_t t0 = 0;
    for (uint32_t i = 1;; ++i) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.flags[a.rank] + base + r) : "memory");
        if ((int32_t)(seen - epoch) >= 0) return true;
        if (i & 0x3FFu) continue;
        if (t0 == 0) { t0 = ar_global_ns(); continue; }
        if (ar_global_ns() - t0 > a.timeout_ns) {
            if (blockIdx.x == 0) printf("nsb exchange: rank %d gave up waiting for rank %d at epoch %u (flag set %d)\n", a.rank, r, epoch, base);
            atomicMax(&g_peer_error, 1u + (unsigned)r);
            return false;
        }
    }
}
__global__ void __launch_bounds__(256) grad_reduce_scatter_kernel(const __grid_constant__ AdamArParams a) {
    const int world = a.world;
    const uint32_t epoch = a.t_dev ? (uint32_t)(*a.t_dev + 1) : a.epoch;
    __shared__ int s_abort, s_timeout;       // s_abort: skip this epoch's update; s_timeout: ... because a peer never arrived
    const uint32_t bad = (a.loss_guard && !isfinite(*a.loss_guard)) ? 1u : 0u;
    if (threadIdx.x == 0) { s_abort = 0; s_timeout = 0; }
    __syncthreads();
    if (threadIdx.x < world) {
        const int r = threadIdx.x;
        const int bad_ofs = world * (1 + (int)(epoch & 1u));
        if (blockIdx.x == 0) {
            asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(a.flags[r] + bad_ofs + a.rank), "r"(bad) : "memory");
            __threadfence_system();
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flags[r] + a.rank), "r"(epoch) : "memory");
        }
        if (!wait_peer_flags(a, 0, r, epoch)) { s_abort = 1; s_timeout = 1; }
        uint32_t peer_bad;
        asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(peer_bad) : "l"(a.flags[a.rank] + bad_ofs + r) : "memory");
        if (peer_bad) s_abort = 1;
    }
    __syncthreads();
    if (!s_abort) {
        const int64_t total4 = (a.n >> 2) * a.n_nets;
        const int64_t per = (total4 + world - 1) / world;
        const int64_t begin = a.rank * per, end = begin + per < total4 ? begin + per : total4;
        for (int64_t i = begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < end; i += (int64_t)gridDim.x * blockDim.x)
            st_mc(reinterpret_cast<float4*>(a.mc_red) + i, ld_reduce_mc(reinterpret_cast<const float4*>(a.mc_grads) + i));
    }
    __threadfence_system();                 // this block's multicast stores are performed before it counts itself done
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_abort) atomicExch(&a.local_sync[1], (int)epoch);        // kernel 2 of this epoch skips the update
        if (s_timeout) atomicExch(&a.local_sync[2], (int)epoch);      // a slice that was never reduced must not be announced
        if (atomicAdd(&a.local_sync[0], 1) == (int)gridDim.x - 1) {   // last block of this rank: publish "my slice is stored"
            a.local_sync[0] = 0;
            __threadfence_system();
            if (*reinterpret_cast<volatile int*>(a.local_sync + 2) != (int)epoch)      // (after a timeout the peers time out too: all raise)
                for (int r = 0; r < world; ++r)
                    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flags[r] + 3 * world + a.rank), "r"(epoch) : "memory");
        }
    }
}
__global__ void __launch_bounds__(256) adam_reduced_kernel(const __grid_constant__ AdamArParams a) {
    const int world = a.world;
    float lr_over_bc1 = a.lr_over_bc1, inv_sqrt_bc2 = a.inv_sqrt_bc2;
    uint32_t epoch = a.epoch;
    if (a.t_dev) { adam_bias_corrections(a.t_dev, a.lr, a.eta_min, a.T_max, a.b1, a.b2, lr_over_bc1, inv_sqrt_bc2); epoch = (uint32_t)(*a.t_dev + 1); }
    __shared__ int s_abort;
    if (threadIdx.x == 0) s_abort = (*reinterpret_cast<volatile int*>(a.local_sync + 1) == (int)epoch) ? 1 : 0;
    __syncthreads();
    if (s_abort) return;
    if (threadIdx.x < world && !wait_peer_flags(a, 3 * world, threadIdx.x, epoch)) s_abort = 1;
    __syncthreads();
    if (s_abort) return;
    const int64_t n4 = a.n >> 2, total4 = n4 * a.n_nets;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / n4);
        const int64_t j = i - k * n4;
        float4 g = ld_peer(reinterpret_cast<const float4*>(a.red) + i);      // written by the peers' multicast stores: not through a stale L1 line
        float4 pm = reinterpret_cast<float4*>(a.m[k])[j], pv = reinterpret_cast<float4*>(a.v[k])[j], pp = reinterpret_cast<float4*>(a.p[k])[j];
        float* gg = &g.x; float* mm = &pm.x; float* vv = &pv.x; float* pq = &pp.x;
#pragma unroll
        for (int c = 0; c < 4; ++c) adam_update(pq[c], mm[c], vv[c], gg[c], a.grad_scale, a.b1, a.b2, a.eps, lr_over_bc1, inv_sqrt_bc2);
        reinterpret_cast<float4*>(a.m[k])[j] = pm; reinterpret_cast<float4*>(a.v[k])[j] = pv; reinterpret_cast<float4*>(a.p[k])[j] = pp;
    }
}

}  // namespace nsb

using namespace nsb;

namespace nsb {
int adam_allreduce_impl(float* const* params, float* const* m, float* const* v, int n_nets, const void* const* peer_grads,
                        void* const* peer_flags, int rank, int world, uint32_t epoch, int64_t n, float lr, float beta1,
                        float beta2, float eps, int64_t t, float grad_scale, const uint64_t* t_dev, float eta_min, int64_t T_max,
                        const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync, const float* loss_guard, void* stream) {
    if (!params || !m || !v || !peer_grads || (!peer_flags && world > 1) || n_nets < 1 || n_nets > kMaxNets || n < 4 || (n & 3) || t < 1 ||
        world < 1 || world > kMaxPeers || rank < 0 || rank >= world)
        return NSB_E_BADARG;
    AdamArParams a{};
    for (int k = 0; k < n_nets; ++k) {
        if (!params[k] || !m[k] || !v[k]) return NSB_E_BADARG;
        a.p[k] = params[k]; a.m[k] = m[k]; a.v[k] = v[k];
    }
    for (int r = 0; r < world; ++r) {
        if (!peer_grads[r] || (world > 1 && !peer_flags[r])) return NSB_E_BADARG;
        a.grads[r] = static_cast<const float*>(peer_grads[r]); a.flags[r] = world > 1 ? static_cast<uint32_t*>(peer_flags[r]) : nullptr;
    }
    const double bc1 = 1.0 - pow((double)beta1, (double)t), bc2 = 1.0 - pow((double)beta2, (double)t);
    a.rank = rank; a.world = world; a.n_nets = n_nets; a.epoch = epoch; a.n = n;
    a.lr_over_bc1 = (float)(lr / bc1); a.b1 = beta1; a.b2 = beta2; a.eps = eps; a.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    a.grad_scale = grad_scale; a.t_dev = t_dev; a.lr = lr; a.eta_min = eta_min; a.T_max = T_max;
    a.mc_grads = static_cast<const float*>(mc_grads);
    a.mc_red = static_cast<float*>(mc_reduced); a.red = reduced; a.local_sync = local_sync;
    a.loss_guard = loss_guard;
    static const uint64_t timeout_ns = [] {
        const char* e = getenv("NSB_PEER_TIMEOUT_S");
        const double sec = e && atof(e) > 0 ? atof(e) : 600.0;
        return (uint64_t)(sec * 1e9);
    }();
    a.timeout_ns = timeout_ns;
    if (world > 1 && mc_grads && mc_reduced && reduced && local_sync) {
        // two-phase exchange through the switch: reduce-scatter + multicast store, then Adam on the local reduced copy
        const int64_t total4 = (n >> 2) * n_nets, per = cdiv(total4, world);
        int g1 = (int)cdiv(per, 256);
        if (g1 > num_sms()) g1 = num_sms();
        grad_reduce_scatter_kernel<<<g1, 256, 0, as_stream(stream)>>>(a);
        NSB_LAUNCH_CHECK("grad_reduce_scatter_kernel");
        int g2 = (int)cdiv(total4, 256);
        if (g2 > 4 * num_sms()) g2 = 4 * num_sms();
        adam_reduced_kernel<<<g2, 256, 0, as_stream(stream)>>>(a);
        NSB_LAUNCH_CHECK("adam_reduced_kernel");
        return NSB_OK;
    }
    // every block spins on the flag exchange first, so the whole grid must be co-resident: cap it at what the occupancy
    // calculator says fits (registers of the chosen instantiation included), at most four blocks per SM
    void (*kern)(const AdamArParams) = world == 1 ? adam_allreduce_kernel<1> : world == 2 ? adam_allreduce_kernel<2>
                                     : world == 4 ? adam_allreduce_kernel<4> : world == 8 ? adam_allreduce_kernel<8> : adam_allreduce_kernel<0>;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0) != cudaSuccess || per_sm < 1) return check_launch("occupancy(adam_allreduce_kernel)");
    if (per_sm > 4) per_sm = 4;
    int grid = (int)cdiv((n >> 2) * n_nets, 256);
    if (grid > per_sm * num_sms()) grid = per_sm * num_sms();
    kern<<<grid, 256, 0, as_stream(stream)>>>(a);
    NSB_LAUNCH_CHECK("adam_allreduce_kernel");
    return NSB_OK;
}
int peer_status(int* code) {
    unsigned int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_peer_error, sizeof(v)) != cudaSuccess) return check_launch("cudaMemcpyFromSymbol(g_peer_error)");
    *code = (int)v;
    return NSB_OK;
}
}  // namespace nsb

extern "C" int nsb_adam_allreduce_step(float* const* params, float* const* m, float* const* v, int n_nets, const void* const* peer_grads,
                                       const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync,
                                       void* const* peer_flags, int rank, int world, uint32_t epoch, int64_t n,
                                       float lr, float beta1, float beta2, float eps, int64_t t, float grad_scale, const float* loss_guard,
                                       void* stream) {
    return adam_allreduce_impl(params, m, v, n_nets, peer_grads, peer_flags, rank, world, epoch, n, lr, beta1, beta2, eps, t, grad_scale,
                               nullptr, 0.f, 0, mc_grads, mc_reduced, reduced, local_sync, loss_guard, stream);
}

extern "C" int nsb_peer_status(int* code) {
    if (!code) return NSB_E_BADARG;
    return peer_status(code);
}

extern "C" int nsb_encode(const float* x, float* out, int64_t Q, int D, int L, int include_input, void* stream) {
    if (Q == 0) return NSB_OK;
    if (!x || !out || Q < 0 || D < 1 || L < 0) return NSB_E_BADARG;
    const int od = D * (include_input ? 1 : 0) + 2 * L * D;
    encode_kernel<<<elem_grid(Q * od), 256, 0, as_stream(stream)>>>(x, out, Q, D, L, include_input);
    NSB_LAUNCH_CHECK("encode_kernel");
    return NSB_OK;
}

extern "C" int nsb_encode_bwd(const float* x, const float* g_out, float* g_x, int64_t Q, int D, int L, int include_input, void* stream) {
    if (Q == 0) return NSB_OK;
    if (!x || !g_out || !g_x || Q < 0 || D < 1 || L < 0) return NSB_E_BADARG;
    encode_bwd_kernel<<<elem_grid(Q * D), 256, 0, as_stream(stream)>>>(x, g_out, g_x, Q, D, L, include_input);
    NSB_LAUNCH_CHECK("encode_bwd_kernel");
    return NSB_OK;
}

extern "C" int nsb_encode_bwd_rays(const float* d_enc_pos, const float* d_enc_dir, const float* rays_o, const float* rays_d, const float* z,
                                   const float* ray_norm, const float* viewdirs, float* d_rays_o, float* d_rays_d, float* d_viewdirs,
                                   int64_t B, int N, void* stream) {
    if (B == 0) return NSB_OK;
    if (!d_enc_pos || !d_enc_dir || !rays_o || !rays_d || !z || B < 0 || N < 1) return NSB_E_BADARG;
    if (!d_rays_o && !d_rays_d && !d_viewdirs) return NSB_E_BADARG;
    encode_bwd_rays_kernel<<<elem_grid(B * 32), 256, 0, as_stream(stream)>>>(d_enc_pos, d_enc_dir, rays_o, rays_d, z, ray_norm, viewdirs,
                                                                          d_rays_o, d_rays_d, d_viewdirs, B, N);
    NSB_LAUNCH_CHECK("encode_bwd_rays_kernel");
    return NSB_OK;
}

namespace nsb {
int adam_impl(float* params, const float* grads, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps, int64_t t,
              float grad_scale, const uint64_t* t_dev, float eta_min, int64_t T_max, const float* loss_guard, void* stream) {
    if (!params || !grads || !m || !v || n < 1 || t < 1) return NSB_E_BADARG;
    const double bc1 = 1.0 - pow((double)beta1, (double)t), bc2 = 1.0 - pow((double)beta2, (double)t);
    adam_kernel<<<elem_grid(n), 256, 0, as_stream(stream)>>>(params, grads, m, v, n, (float)(lr / bc1), beta1, beta2, eps,
                                                            (float)(1.0 / sqrt(bc2)), grad_scale, t_dev, lr, eta_min, T_max, loss_guard);
    NSB_LAUNCH_CHECK("adam_kernel");
    return NSB_OK;
}
}  // namespace nsb

extern "C" int nsb_adam_step(float* params, const float* grads, float* m, float* v, int64_t n, float lr, float beta1,
                             float beta2, float eps, int64_t t, float grad_scale, const float* loss_guard, void* stream) {
    return adam_impl(params, grads, m, v, n, lr, beta1, beta2, eps, t, grad_scale, nullptr, 0.f, 0, loss_guard, stream);
}

// ---- torch.nn.utils.clip_grad_norm_ (train/trainer.py:719-721) on the flat gradient buffer -------------------------------
namespace nsb {
__global__ void grad_sumsq_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ acc) {
    float s = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s = fmaf(g[i], g[i], s);
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) atomicAdd(acc, s);
}
__global__ void grad_clip_kernel(float* __restrict__ g, int64_t n, const float* __restrict__ acc, float max_norm, float pre_scale) {
    // total_norm of (pre_scale * g); clip_coef = max_norm / (total_norm + 1e-6), clamped to 1 (torch semantics)
    const float coef = fminf(max_norm / (sqrtf(*acc) * pre_scale + 1e-6f), 1.0f);
    if (coef >= 1.0f) return;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) g[i] *= coef;
}
}  // namespace nsb

extern "C" int nsb_grad_clip(float* grads, int64_t n, float max_norm, float pre_scale, float* scratch, void* stream) {
    if (!grads || !scratch || n < 1 || !(max_norm > 0.f)) return NSB_E_BADARG;
    cudaStream_t st = as_stream(stream);
    if (cudaMemsetAsync(scratch, 0, sizeof(float), st) != cudaSuccess) return NSB_E_CUDA;
    grad_sumsq_kernel<<<elem_grid(n), 256, 0, st>>>(grads, n, scratch);
    NSB_LAUNCH_CHECK("grad_sumsq_kernel");
    grad_clip_kernel<<<elem_grid(n), 256, 0, st>>>(grads, n, scratch, max_norm, pre_scale);
    NSB_LAUNCH_CHECK("grad_clip_kernel");
    return NSB_OK;
}
