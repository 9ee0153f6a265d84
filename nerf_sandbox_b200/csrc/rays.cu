// Camera-ray generation + NDC warp (SURVEY section 8f rank 1): utils/ray_utils.py:10-136.
// One thread per pixel, everything in registers, six coalesced outputs.  Compiled -fmad=false so each
// mul/add/div rounds like the reference's separate ATen ops.
#include "nsb_common.cuh"

namespace nsb {

struct RayCam {
    float fx, fy, cx, cy;
    float R[9];      // row-major c2w[:3,:3]
    float t[3];      // c2w[:3,3]
    float sy_cam, sz_cam;   // camera-frame signs of (y, z): opengl (-1,-1), opencv (+1,+1), pytorch3d (-1,+1)  (:69-77)
};

struct RayOut { float ow[3], du[3], nrm, om[3], dm[3], nm; };

// one pixel -> the reference's six outputs (ray_utils.py:62-126)
__device__ __forceinline__ RayOut ray_from_pixel(const RayCam& c, float x, float y, int H, int W, int pixel_center, int as_ndc,
                                                float near_plane) {
    RayOut o;
    if (pixel_center) { x += 0.5f; y += 0.5f; }
    const float xc = (x - c.cx) / c.fx, yc = (y - c.cy) / c.fy;                // :66-67
    const float dc[3] = {xc, c.sy_cam * yc, c.sz_cam};
    float d[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) d[r] = dc[0] * c.R[3 * r] + dc[1] * c.R[3 * r + 1] + dc[2] * c.R[3 * r + 2];   // dirs @ R^T :80
    const float nrm = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);          // :81
    const float inv = nrm + 1e-9f;
#pragma unroll
    for (int r = 0; r < 3; ++r) { o.ow[r] = c.t[r]; o.du[r] = d[r] / inv; }    // :82-83
    o.nrm = nrm;
    if (!as_ndc) {                                                             // :86-90
#pragma unroll
        for (int r = 0; r < 3; ++r) { o.om[r] = c.t[r]; o.dm[r] = o.du[r]; }
        o.nm = nrm;
    } else {                                                                   // :92-126
        const float sx = 2.0f * c.fx / (float)W, sy = 2.0f * c.fx / (float)H;  // scalar focal = fx (:100-102)
        const float tn = -(near_plane + c.t[2]) / (d[2] + 1e-9f);              // :108
        const float ow[3] = {c.t[0] + tn * d[0], c.t[1] + tn * d[1], c.t[2] + tn * d[2]};
        const float oz = ow[2] + 1e-9f, dz = d[2] + 1e-9f;
        o.om[0] = -sx * (ow[0] / oz); o.om[1] = -sy * (ow[1] / oz); o.om[2] = 1.0f + 2.0f * near_plane / oz;   // :112-114
        const float d0 = -sx * (d[0] / dz - ow[0] / oz), d1 = -sy * (d[1] / dz - ow[1] / oz), d2 = -2.0f * near_plane / oz;
        const float nn = sqrtf(d0 * d0 + d1 * d1 + d2 * d2);                   // :125
        const float dn = fmaxf(nn, 1e-12f);                                    // F.normalize :126
        o.dm[0] = d0 / dn; o.dm[1] = d1 / dn; o.dm[2] = d2 / dn;
        o.nm = nn;
    }
    return o;
}

__device__ __forceinline__ void store_ray(const RayOut& o, int64_t i, float* o_world, float* d_world_unit, float* d_world_norm,
                                          float* o_march, float* d_march_unit, float* d_march_norm) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        o_world[3 * i + r] = o.ow[r]; d_world_unit[3 * i + r] = o.du[r]; o_march[3 * i + r] = o.om[r]; d_march_unit[3 * i + r] = o.dm[r];
    }
    d_world_norm[i] = o.nrm; d_march_norm[i] = o.nm;
}

__global__ void camera_rays_kernel(RayCam c, int H, int W, const float* __restrict__ pixels_xy, int64_t n, int pixel_center,
                                   int as_ndc, float near_plane, float* __restrict__ o_world, float* __restrict__ d_world_unit,
                                   float* __restrict__ d_world_norm, float* __restrict__ o_march, float* __restrict__ d_march_unit,
                                   float* __restrict__ d_march_norm) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float x, y;
        if (pixels_xy) { x = pixels_xy[2 * i]; y = pixels_xy[2 * i + 1]; }        // :56-60
        else { x = (float)(i % W); y = (float)(i / W); }                           // :45-54 (row-major meshgrid)
        store_ray(ray_from_pixel(c, x, y, H, W, pixel_center, as_ndc, near_plane), i, o_world, d_world_unit, d_world_norm, o_march,
                  d_march_unit, d_march_norm);
    }
}

// Device-side pixel batch sampler (SURVEY section 8f rank 2): data/samplers.py:134-290 without the host round trips.
// Per ray: frame id (fixed, or uniform when fid < 0), pixel uniform in the crop window (:119-127), RGBA -> white composite
// (:129-132), rays with pixel_center=True (:181-188).
__global__ void sample_pixel_batch_kernel(const float* __restrict__ images, int F, int H, int W, int C, const float* __restrict__ Ks,
                                          const float* __restrict__ c2ws, int fid, int h0, int h1, int w0, int w1, int white_bkgd,
                                          float sy_cam, float sz_cam, int as_ndc, float near_plane, int64_t B, uint64_t seed,
                                          uint64_t step, float* __restrict__ rgb, float* __restrict__ pixels_xy,
                                          int* __restrict__ fids_out, float* __restrict__ o_world, float* __restrict__ d_world_unit,
                                          float* __restrict__ d_world_norm, float* __restrict__ o_march,
                                          float* __restrict__ d_march_unit, float* __restrict__ d_march_norm) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < B; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 rnd = philox4(seed, step, (uint64_t)i);
        const int f = fid >= 0 ? fid : min((int)(u01(rnd.z) * (float)F), F - 1);
        const int x = min(w0 + (int)(u01(rnd.x) * (float)(w1 - w0)), w1 - 1);
        const int y = min(h0 + (int)(u01(rnd.y) * (float)(h1 - h0)), h1 - 1);
        const float* px = images + (((size_t)f * H + y) * W + x) * C;
        float r = px[0], g = px[1], b = px[2];
        if (white_bkgd && C == 4) { const float a = px[3]; r = r * a + (1.0f - a); g = g * a + (1.0f - a); b = b * a + (1.0f - a); }
        rgb[3 * i] = r; rgb[3 * i + 1] = g; rgb[3 * i + 2] = b;
        if (pixels_xy) { pixels_xy[2 * i] = (float)x; pixels_xy[2 * i + 1] = (float)y; }
        if (fids_out) fids_out[i] = f;
        RayCam c;
        c.fx = Ks[4 * f]; c.fy = Ks[4 * f + 1]; c.cx = Ks[4 * f + 2]; c.cy = Ks[4 * f + 3];
#pragma unroll
        for (int rr = 0; rr < 3; ++rr) {
#pragma unroll
            for (int k = 0; k < 3; ++k) c.R[3 * rr + k] = c2ws[12 * f + 4 * rr + k];
            c.t[rr] = c2ws[12 * f + 4 * rr + 3];
        }
        c.sy_cam = sy_cam; c.sz_cam = sz_cam;
        store_ray(ray_from_pixel(c, (float)x, (float)y, H, W, 1, as_ndc, near_plane), i, o_world, d_world_unit, d_world_norm, o_march,
                  d_march_unit, d_march_norm);
    }
}

// ---- camera-ray backward: d(six outputs) -> d c2w[:3,:4] per frame (pose refinement, iNeRF / BARF) ----
// Per ray, the forward of ray_from_pixel is recomputed in registers with the same expressions (this file is compiled with
// -fmad=false, so the recomputed intermediates are bitwise the forward's), then differentiated by hand:
//   d = R dc,  nrm = |d|,  du = d / (nrm + 1e-9)                                   (world outputs; o_world = t)
//   NDC: tn = -(near + t_z) / (d_z + 1e-9), ow = t + tn d, oz = ow_z + 1e-9, dz = d_z + 1e-9, om / D as the forward,
//        nn = |D|, dm = D / max(nn, 1e-12)                                          (F.normalize's backward)
// and dL/dR[r][k] = dL/dd_r * dc_k, dL/dt_r.  Rays are summed into their frame's 12-vector without atomics: each block owns
// one [F,12] slice of block partials in the workspace and adds its tiles of 256 rays to it in tile order (one warp per
// (frame, component) pair, a fixed butterfly over the tile); camera_rays_bwd_reduce_kernel then sums the block partials in
// block order.  The result is bitwise repeatable, and a frame no ray belongs to gets exactly zero.
struct RayGrad { const float *ow, *du, *nrm, *om, *dm, *nm; };

constexpr int kRaysBwdThreads = 256;
constexpr int kRaysBwdMaxBlocks = 296;
static inline int rays_bwd_blocks(int64_t n) { return (int)(cdiv(n, kRaysBwdThreads) < kRaysBwdMaxBlocks ? cdiv(n, kRaysBwdThreads) : kRaysBwdMaxBlocks); }

__device__ __forceinline__ float opt_ld(const float* p, int64_t i) { return p ? p[i] : 0.0f; }

__device__ __forceinline__ void ray_bwd_from_pixel(const RayCam& c, float x, float y, int H, int W, int pixel_center, int as_ndc,
                                                   float near_plane, const RayGrad& g, int64_t i, float out[12]) {
    if (pixel_center) { x += 0.5f; y += 0.5f; }
    const float xc = (x - c.cx) / c.fx, yc = (y - c.cy) / c.fy;
    const float dc[3] = {xc, c.sy_cam * yc, c.sz_cam};
    float d[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) d[r] = dc[0] * c.R[3 * r] + dc[1] * c.R[3 * r + 1] + dc[2] * c.R[3 * r + 2];
    const float nrm = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    const float inv = nrm + 1e-9f;
    float gd[3] = {0.f, 0.f, 0.f}, gt[3], gdu[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) { gt[r] = opt_ld(g.ow, 3 * i + r); gdu[r] = opt_ld(g.du, 3 * i + r); }
    float gnrm = opt_ld(g.nrm, i);
    if (!as_ndc) {                                             // marching rays are the world rays
#pragma unroll
        for (int r = 0; r < 3; ++r) { gt[r] += opt_ld(g.om, 3 * i + r); gdu[r] += opt_ld(g.dm, 3 * i + r); }
        gnrm += opt_ld(g.nm, i);
    } else {
        const float sx = 2.0f * c.fx / (float)W, sy = 2.0f * c.fx / (float)H;
        const float e = d[2] + 1e-9f;
        const float tn = -(near_plane + c.t[2]) / e;
        const float ow[3] = {c.t[0] + tn * d[0], c.t[1] + tn * d[1], c.t[2] + tn * d[2]};
        const float oz = ow[2] + 1e-9f, dz = e;
        const float D[3] = {-sx * (d[0] / dz - ow[0] / oz), -sy * (d[1] / dz - ow[1] / oz), -2.0f * near_plane / oz};
        const float nn = sqrtf(D[0] * D[0] + D[1] * D[1] + D[2] * D[2]);
        const float dn = fmaxf(nn, 1e-12f);
        const float gdm[3] = {opt_ld(g.dm, 3 * i), opt_ld(g.dm, 3 * i + 1), opt_ld(g.dm, 3 * i + 2)};
        const float gom[3] = {opt_ld(g.om, 3 * i), opt_ld(g.om, 3 * i + 1), opt_ld(g.om, 3 * i + 2)};
        // dm = D / max(nn, eps), nm = nn
        const float gD_dot = gdm[0] * D[0] + gdm[1] * D[1] + gdm[2] * D[2];
        const float kD = nn > 0.f ? (opt_ld(g.nm, i) - (nn > 1e-12f ? gD_dot / (dn * dn) : 0.f)) / nn : 0.f;
        float gD[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) gD[r] = gdm[r] / dn + D[r] * kD;
        const float s[2] = {sx, sy};
        const float oz2 = oz * oz;
        float gow[3] = {0.f, 0.f, 0.f}, goz = 0.f, gdz = 0.f;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            // D_r = -s (d_r / dz - ow_r / oz),  om_r = -s ow_r / oz
            gd[r] += -s[r] * gD[r] / dz;
            gdz += s[r] * gD[r] * d[r] / (dz * dz);
            gow[r] += s[r] * (gD[r] - gom[r]) / oz;
            goz += s[r] * (gom[r] - gD[r]) * ow[r] / oz2;
        }
        goz += 2.0f * near_plane * (gD[2] - gom[2]) / oz2;     // D_2 = -2 near / oz,  om_2 = 1 + 2 near / oz
        gow[2] += goz;
        gd[2] += gdz;
        // ow = t + tn d,  tn = -(near + t_z) / e
        const float gtn = gow[0] * d[0] + gow[1] * d[1] + gow[2] * d[2];
#pragma unroll
        for (int r = 0; r < 3; ++r) { gt[r] += gow[r]; gd[r] += tn * gow[r]; }
        gt[2] += -gtn / e;
        gd[2] += gtn * (near_plane + c.t[2]) / (e * e);
    }
    // du = d / (nrm + 1e-9),  nrm = |d|
    const float gdu_d = gdu[0] * d[0] + gdu[1] * d[1] + gdu[2] * d[2];
    gnrm += -gdu_d / (inv * inv);
    const float kn = nrm > 0.f ? gnrm / nrm : 0.f;
#pragma unroll
    for (int r = 0; r < 3; ++r) gd[r] += gdu[r] / inv + d[r] * kn;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int k = 0; k < 3; ++k) out[4 * r + k] = gd[r] * dc[k];
        out[4 * r + 3] = gt[r];
    }
}

__global__ void __launch_bounds__(kRaysBwdThreads)
camera_rays_bwd_kernel(int H, int W, const float* __restrict__ Ks, const float* __restrict__ c2ws, int F, const int* __restrict__ fids,
                       float sy_cam, float sz_cam, int pixel_center, int as_ndc, float near_plane, const float* __restrict__ pixels_xy,
                       int64_t n, RayGrad g, float* __restrict__ partial) {
    __shared__ float vals[12][kRaysBwdThreads];
    __shared__ int tile_fid[kRaysBwdThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kRaysBwdThreads / 32;
    const int pairs = 12 * F;
    float* mine = partial + (int64_t)blockIdx.x * pairs;
    if (lane == 0)
        for (int p = warp; p < pairs; p += nwarps) mine[p] = 0.f;
    const int64_t tiles = (n + kRaysBwdThreads - 1) / kRaysBwdThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = tile * kRaysBwdThreads + tid;
        int f = -1;
        float out[12];
        if (i < n) {
            f = fids ? fids[i] : 0;
            if (f < 0 || f >= F) f = -1;                       // a ray of no frame contributes nothing
        }
        if (f >= 0) {
            float x, y;
            if (pixels_xy) { x = pixels_xy[2 * i]; y = pixels_xy[2 * i + 1]; }
            else { x = (float)(i % W); y = (float)(i / W); }
            RayCam c;
            c.fx = Ks[4 * f]; c.fy = Ks[4 * f + 1]; c.cx = Ks[4 * f + 2]; c.cy = Ks[4 * f + 3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int k = 0; k < 3; ++k) c.R[3 * r + k] = c2ws[12 * f + 4 * r + k];
                c.t[r] = c2ws[12 * f + 4 * r + 3];
            }
            c.sy_cam = sy_cam; c.sz_cam = sz_cam;
            ray_bwd_from_pixel(c, x, y, H, W, pixel_center, as_ndc, near_plane, g, i, out);
        } else {
#pragma unroll
            for (int k = 0; k < 12; ++k) out[k] = 0.f;
        }
#pragma unroll
        for (int k = 0; k < 12; ++k) vals[k][tid] = out[k];
        tile_fid[tid] = f;
        __syncthreads();
        for (int p = warp; p < pairs; p += nwarps) {
            const int pf = p / 12, pc = p - 12 * pf;
            float s = 0.f;
            bool hit = false;
#pragma unroll
            for (int k = lane; k < kRaysBwdThreads; k += 32)
                if (tile_fid[k] == pf) { s += vals[pc][k]; hit = true; }
            if (__any_sync(0xffffffffu, hit)) {
                s = warp_sum(s);
                if (lane == 0) mine[p] += s;
            }
        }
        __syncthreads();
    }
}

// d_c2ws[p] = sum over blocks of partial[block][p], block order; one warp per (frame, component)
__global__ void camera_rays_bwd_reduce_kernel(const float* __restrict__ partial, int blocks, int pairs, float* __restrict__ d_c2ws) {
    const int lane = threadIdx.x & 31;
    const int p = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    if (p >= pairs) return;
    float s = 0.f;
    for (int b = lane; b < blocks; b += 32) s += partial[(int64_t)b * pairs + p];
    s = warp_sum(s);
    if (lane == 0) d_c2ws[p] = s;
}

// ---- eval output path (SURVEY 8f rank 4): what validation_renderer.py:485-533 + render_utils.py:28-47 do with a frame ----
// u8 = (clamp(x, 0, 1) * 255 + 0.5) truncated  (two roundings: this file is compiled with -fmad=false, like numpy)
__device__ __forceinline__ uint8_t to_u8(float x) { return (uint8_t)(fminf(fmaxf(x, 0.0f), 1.0f) * 255.0f + 0.5f); }
__global__ void frame_output_kernel(const float* __restrict__ rgb, const float* __restrict__ acc, const float* __restrict__ depth, int64_t n,
                                    float near_, float range, int use_ndc, uint8_t* __restrict__ rgb8, uint8_t* __restrict__ acc8,
                                    uint8_t* __restrict__ depth8, const float* __restrict__ gt, const float* __restrict__ mask,
                                    double* __restrict__ psnr_acc) {
    double se = 0.0, wsum = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float r = rgb[3 * i], g = rgb[3 * i + 1], b = rgb[3 * i + 2];
        if (rgb8) { rgb8[3 * i] = to_u8(r); rgb8[3 * i + 1] = to_u8(g); rgb8[3 * i + 2] = to_u8(b); }
        if (acc8 && acc) acc8[i] = to_u8(acc[i]);
        // :491-492 -- a true IEEE division by fp32(far - near + 1e-8), as torch's `tensor / python_float` does: byte-exact
        if (depth8 && depth) depth8[i] = to_u8(use_ndc ? depth[i] : (depth[i] - near_) / range);
        if (gt && psnr_acc) {                                                                           // _compute_psnr, :171-196
            const float m = mask ? mask[i] : 1.0f;
            float e = 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float d = fminf(fmaxf(rgb[3 * i + c], 0.0f), 1.0f) - fminf(fmaxf(gt[3 * i + c], 0.0f), 1.0f);
                e += d * d;
            }
            se += (double)(e * m); wsum += (double)m;
        }
    }
    if (gt && psnr_acc) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { se += __shfl_xor_sync(0xffffffffu, se, d); wsum += __shfl_xor_sync(0xffffffffu, wsum, d); }
        if ((threadIdx.x & 31) == 0) { atomicAdd(psnr_acc, se); atomicAdd(psnr_acc + 1, wsum); }
    }
}
__global__ void psnr_finish_kernel(const double* __restrict__ acc, float* __restrict__ out) {
    // mse = sum(diff^2 * m) / max(sum(m) * 3, 1e-8);  psnr = -10 log10(max(mse, 1e-10))
    const double denom = acc[1] * 3.0 > 1e-8 ? acc[1] * 3.0 : 1e-8;
    const double mse = acc[0] / denom;
    out[0] = (float)(-10.0 * log10(mse > 1e-10 ? mse : 1e-10));
    out[1] = (float)mse;
}

}  // namespace nsb

using namespace nsb;

extern "C" int nsb_frame_output(const float* rgb, const float* acc, const float* depth, int64_t n, double depth_near, double depth_far,
                                int use_ndc, uint8_t* rgb8, uint8_t* acc8, uint8_t* depth8, const float* gt_rgb, const float* mask,
                                double* psnr_scratch, float* psnr_out, void* stream) {
    if (n == 0) return NSB_OK;
    if (!rgb || n < 0) return NSB_E_BADARG;
    if (gt_rgb && (!psnr_scratch || !psnr_out)) return NSB_E_BADARG;
    cudaStream_t st = as_stream(stream);
    if (gt_rgb && cudaMemsetAsync(psnr_scratch, 0, 2 * sizeof(double), st) != cudaSuccess) return NSB_E_CUDA;
    const int64_t want = cdiv(n, 256), cap = (int64_t)num_sms() * 8;
    // Python evaluates `far - near + 1e-8` in double and torch rounds that scalar to the tensor's dtype
    const float range = (float)(depth_far - depth_near + 1e-8);
    frame_output_kernel<<<(int)(want < cap ? want : cap), 256, 0, st>>>(rgb, acc, depth, n, (float)depth_near, range, use_ndc, rgb8, acc8, depth8,
                                                                       gt_rgb, mask, gt_rgb ? psnr_scratch : nullptr);
    NSB_LAUNCH_CHECK("frame_output_kernel");
    if (gt_rgb) {
        psnr_finish_kernel<<<1, 1, 0, st>>>(psnr_scratch, psnr_out);
        NSB_LAUNCH_CHECK("psnr_finish_kernel");
    }
    return NSB_OK;
}

extern "C" int nsb_camera_rays(int H, int W, const float* K_host, const float* c2w_host, int c2w_cols, int convention,
                               int pixel_center, int as_ndc, float near_plane, const float* pixels_xy, int64_t n_pixels,
                               float* o_world, float* d_world_unit, float* d_world_norm, float* o_march, float* d_march_unit,
                               float* d_march_norm, void* stream) {
    if (!K_host || !c2w_host || (c2w_cols != 4) || H < 1 || W < 1 || convention < 0 || convention > 2) return NSB_E_BADARG;
    const int64_t n = pixels_xy ? n_pixels : (int64_t)H * W;
    if (n == 0) return NSB_OK;
    if (!o_world || !d_world_unit || !d_world_norm || !o_march || !d_march_unit || !d_march_norm) return NSB_E_BADARG;
    RayCam c;
    c.fx = K_host[0]; c.fy = K_host[4]; c.cx = K_host[2]; c.cy = K_host[5];
    for (int r = 0; r < 3; ++r) { for (int k = 0; k < 3; ++k) c.R[3 * r + k] = c2w_host[4 * r + k]; c.t[r] = c2w_host[4 * r + 3]; }
    c.sy_cam = convention == 1 ? 1.0f : -1.0f;
    c.sz_cam = convention == 0 ? -1.0f : 1.0f;
    const int64_t want = cdiv(n, 256), cap = (int64_t)num_sms() * 16;
    camera_rays_kernel<<<(int)(want < cap ? want : cap), 256, 0, as_stream(stream)>>>(
        c, H, W, pixels_xy, n, pixel_center, as_ndc, near_plane, o_world, d_world_unit, d_world_norm, o_march, d_march_unit, d_march_norm);
    NSB_LAUNCH_CHECK("camera_rays_kernel");
    return NSB_OK;
}

extern "C" size_t nsb_camera_rays_bwd_workspace_bytes(int64_t n, int F) {
    if (n <= 0 || F < 1) return 0;
    return align_up((size_t)rays_bwd_blocks(n) * 12 * (size_t)F * sizeof(float), 256);
}

extern "C" int nsb_camera_rays_bwd(int H, int W, const float* Ks, const float* c2ws, int F, const int* fids, int convention,
                                   int pixel_center, int as_ndc, float near_plane, const float* pixels_xy, int64_t n,
                                   const float* g_o_world, const float* g_d_world_unit, const float* g_d_world_norm,
                                   const float* g_o_march, const float* g_d_march_unit, const float* g_d_march_norm,
                                   float* d_c2ws, void* ws, size_t ws_bytes, void* stream) {
    if (!Ks || !c2ws || !d_c2ws || F < 1 || H < 1 || W < 1 || n < 0 || convention < 0 || convention > 2) return NSB_E_BADARG;
    if (!g_o_world && !g_d_world_unit && !g_d_world_norm && !g_o_march && !g_d_march_unit && !g_d_march_norm) return NSB_E_BADARG;
    if (!pixels_xy && n != (int64_t)H * W) return NSB_E_BADARG;
    cudaStream_t st = as_stream(stream);
    if (n == 0)
        return cudaMemsetAsync(d_c2ws, 0, (size_t)F * 12 * sizeof(float), st) == cudaSuccess ? NSB_OK : NSB_E_CUDA;
    if (!ws) return NSB_E_BADARG;
    if (ws_bytes < nsb_camera_rays_bwd_workspace_bytes(n, F)) return NSB_E_WORKSPACE;
    const int blocks = rays_bwd_blocks(n), pairs = 12 * F;
    float* partial = static_cast<float*>(ws);
    const RayGrad g{g_o_world, g_d_world_unit, g_d_world_norm, g_o_march, g_d_march_unit, g_d_march_norm};
    camera_rays_bwd_kernel<<<blocks, kRaysBwdThreads, 0, st>>>(H, W, Ks, c2ws, F, fids, convention == 1 ? 1.0f : -1.0f,
                                                               convention == 0 ? -1.0f : 1.0f, pixel_center, as_ndc, near_plane,
                                                               pixels_xy, n, g, partial);
    NSB_LAUNCH_CHECK("camera_rays_bwd_kernel");
    camera_rays_bwd_reduce_kernel<<<(int)cdiv((int64_t)pairs * 32, 256), 256, 0, st>>>(partial, blocks, pairs, d_c2ws);
    NSB_LAUNCH_CHECK("camera_rays_bwd_reduce_kernel");
    return NSB_OK;
}

extern "C" int nsb_sample_pixel_batch(const float* images, int F, int H, int W, int C, const float* Ks, const float* c2ws, int fid,
                                      int h0, int h1, int w0, int w1, int white_bkgd, int convention, int as_ndc, float near_plane,
                                      int64_t B, uint64_t seed, uint64_t step, float* rgb, float* pixels_xy, int* fids_out,
                                      float* o_world, float* d_world_unit, float* d_world_norm, float* o_march, float* d_march_unit,
                                      float* d_march_norm, void* stream) {
    if (B == 0) return NSB_OK;
    if (!images || !Ks || !c2ws || !rgb || F < 1 || fid >= F || (C != 3 && C != 4) || convention < 0 || convention > 2) return NSB_E_BADARG;
    if (h0 < 0 || h1 > H || w0 < 0 || w1 > W || h0 >= h1 || w0 >= w1) return NSB_E_BADARG;
    if (!o_world || !d_world_unit || !d_world_norm || !o_march || !d_march_unit || !d_march_norm) return NSB_E_BADARG;
    const int64_t want = cdiv(B, 256), cap = (int64_t)num_sms() * 16;
    sample_pixel_batch_kernel<<<(int)(want < cap ? want : cap), 256, 0, as_stream(stream)>>>(
        images, F, H, W, C, Ks, c2ws, fid, h0, h1, w0, w1, white_bkgd, convention == 1 ? 1.0f : -1.0f, convention == 0 ? -1.0f : 1.0f,
        as_ndc, near_plane, B, seed, step, rgb, pixels_xy, fids_out, o_world, d_world_unit, d_world_norm, o_march, d_march_unit, d_march_norm);
    NSB_LAUNCH_CHECK("sample_pixel_batch_kernel");
    return NSB_OK;
}
