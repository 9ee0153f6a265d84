// Library core + whole-path entry points: the host-side sequencing of Trainer._train_step
// (train/trainer.py:876-1013, + backward) and of one ray tile of render_image_chunked
// (utils/render_utils.py:337-417) as back-to-back launches on one stream -- no host syncs, no
// allocation, so a caller can capture a step in a CUDA graph.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include "nsb_common.cuh"

namespace nsb {

int64_t g_launches = 0;
char g_cuda_err[256] = "";

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
        return NSB_E_CUDA;
    }
    return NSB_OK;
}

int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

// field_fp32.cu
size_t fp32_workspace_bytes(int64_t Q, int stash);
int pack_fp32(const float* params, void* packed, cudaStream_t st);
int fp32_prepare_rays(const float*, const float*, const float*, const float*, const float*, void*, int64_t, int, cudaStream_t);
int fp32_prepare_enc(const float*, const float*, void*, int64_t, cudaStream_t);
int fp32_mlp_fwd(const void* packed, float* raw, void* ws, int64_t Q, cudaStream_t st);
int fp32_mlp_bwd(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws, int64_t Q,
                 cudaStream_t st);
// field_tc.cu
size_t tc_workspace_bytes(int64_t Q, int stash);
size_t tc_stash_tile_bytes();
thread_local const uint64_t* g_step_dev = nullptr;
thread_local uint64_t* g_pack_counter = nullptr;      // nsb_train_step: step counter the next tc_pack launch increments when it is done
int tc_pack(const float* const* params, void* const* packed_bf16, int n_nets, bool train_only, cudaStream_t st);
int tc_field_fwd_rays(const float*, const float*, const float*, const float*, const float*, const void* packed,
                      float* raw, void* ws, int64_t B, int N, int stash, cudaStream_t st);
int tc_field_fwd_enc(const float* enc_pos, const float* enc_dir, const void* packed, float* raw, void* ws, int64_t Q,
                     int stash, cudaStream_t st);
int tc_field_bwd(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws, int64_t Q,
                 cudaStream_t st);

// The fp32 parity mode's INFERENCE forward (no stash) runs on the tensor cores with fp16-split operands (field_tc.cu:
// field_fwd_split_kernel, fp32-accurate).
int tc_field_fwd_rays_split(const float*, const float*, const float*, const float*, const float*, const void* packed, float* raw,
                            int64_t B, int N, cudaStream_t st);
int tc_field_fwd_enc_split(const float* enc_pos, const float* enc_dir, const void* packed, float* raw, int64_t Q, cudaStream_t st);

int composite_raw_fwd_at(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm, float* comp,
                         float* weights, float* acc, float* depth, int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset,
                         int64_t idx0, void* stream);
int tc_debug_layer(const float*, const float*, const float*, const float*, const float*, const void*, float*, float*, int,
                   int64_t, int, cudaStream_t);

static size_t field_ws(int64_t Q, int mode, int stash) {
    return mode == NSB_MODE_BF16 ? tc_workspace_bytes(Q, stash) : fp32_workspace_bytes(Q, stash);
}

}  // namespace nsb

using namespace nsb;

extern "C" int nsb_version(void) { return 100; }
extern "C" const char* nsb_error_string(int code) {
    switch (code) {
        case NSB_OK: return "ok";
        case NSB_E_BADARG: return "bad argument (shape/flag not supported by this path)";
        case NSB_E_WORKSPACE: return "workspace too small";
        case NSB_E_CUDA: return "CUDA error (see nsb_last_cuda_error)";
        case NSB_E_ARCH: return "device is not sm_100";
        default: return "unknown error";
    }
}
extern "C" const char* nsb_last_cuda_error(void) { return g_cuda_err; }
extern "C" int64_t nsb_launch_count(void) { return g_launches; }

extern "C" size_t nsb_packed_weights_bytes(void) { return packed_layout().total; }
extern "C" int nsb_pack_weights_batch(const float* const* params, void* const* packed, int n_nets, int mode, void* stream) {
    bool train_only = false;
    if (mode >= 0 && (mode & NSB_PACK_TRAIN_ONLY)) { train_only = true; mode &= ~NSB_PACK_TRAIN_ONLY; }
    if (!params || !packed || n_nets < 1 || n_nets > 4 || mode < -1 || mode > NSB_MODE_BF16) return NSB_E_BADARG;
    void* bf16[4];
    for (int i = 0; i < n_nets; ++i) {
        if (!params[i] || !packed[i]) return NSB_E_BADARG;
        bf16[i] = reinterpret_cast<char*>(packed[i]) + packed_layout().bf16_off;
        if (mode != NSB_MODE_BF16) NSB_TRY(pack_fp32(params[i], packed[i], as_stream(stream)));
    }
    // one launch for all nets and images; the fp32 mode needs the tensor-core images too (split-operand inference forward)
    if (mode != NSB_MODE_FP32) NSB_TRY(tc_pack(params, bf16, n_nets, train_only, as_stream(stream)));
    else if (!train_only) NSB_TRY(tc_pack(params, bf16, n_nets, false, as_stream(stream)));
    return NSB_OK;
}

extern "C" int nsb_pack_weights(const float* params, void* packed, int mode, void* stream) {
    return nsb_pack_weights_batch(&params, &packed, 1, mode, stream);
}

extern "C" size_t nsb_field_workspace_bytes(int64_t Q, int mode, int stash) { return field_ws(Q, mode, stash); }

extern "C" int nsb_field_fwd_enc(const float* enc_pos, const float* enc_dir, const void* packed, float* raw, void* ws,
                                 size_t ws_bytes, int64_t Q, int mode, int stash, void* stream) {
    if (Q == 0) return NSB_OK;
    if (!enc_pos || !enc_dir || !packed || !raw || !ws || Q < 0) return NSB_E_BADARG;
    if (ws_bytes < field_ws(Q, mode, stash)) return NSB_E_WORKSPACE;
    if (mode == NSB_MODE_BF16)
        return tc_field_fwd_enc(enc_pos, enc_dir, reinterpret_cast<const char*>(packed) + packed_layout().bf16_off, raw,
                                ws, Q, stash, as_stream(stream));
    if (!stash)
        return tc_field_fwd_enc_split(enc_pos, enc_dir, reinterpret_cast<const char*>(packed) + packed_layout().bf16_off, raw, Q, as_stream(stream));
    NSB_TRY(fp32_prepare_enc(enc_pos, enc_dir, ws, Q, as_stream(stream)));
    return fp32_mlp_fwd(packed, raw, ws, Q, as_stream(stream));
}

extern "C" int nsb_field_fwd_rays(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm,
                                  const float* viewdirs, const void* packed, float* raw, void* ws, size_t ws_bytes,
                                  int64_t B, int N, int mode, int stash, void* stream) {
    if (B == 0) return NSB_OK;
    if (!rays_o || !rays_d || !z || !packed || !raw || !ws || B < 0 || N < 1) return NSB_E_BADARG;
    const int64_t Q = B * (int64_t)N;
    if (ws_bytes < field_ws(Q, mode, stash)) return NSB_E_WORKSPACE;
    if (mode == NSB_MODE_BF16)
        return tc_field_fwd_rays(rays_o, rays_d, z, ray_norm, viewdirs,
                                 reinterpret_cast<const char*>(packed) + packed_layout().bf16_off, raw, ws, B, N, stash,
                                 as_stream(stream));
    if (!stash)
        return tc_field_fwd_rays_split(rays_o, rays_d, z, ray_norm, viewdirs, reinterpret_cast<const char*>(packed) + packed_layout().bf16_off, raw,
                                       B, N, as_stream(stream));
    NSB_TRY(fp32_prepare_rays(rays_o, rays_d, z, ray_norm, viewdirs, ws, B, N, as_stream(stream)));
    return fp32_mlp_fwd(packed, raw, ws, Q, as_stream(stream));
}

extern "C" int nsb_field_bwd_ex(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws,
                                size_t ws_bytes, int64_t Q, int mode, void* stream) {
    if (Q == 0) return NSB_OK;
    if (!d_raw || !packed || !ws || Q < 0 || (!grads && !d_enc_pos && !d_enc_dir)) return NSB_E_BADARG;
    if (ws_bytes < field_ws(Q, mode, 1)) return NSB_E_WORKSPACE;
    if (mode == NSB_MODE_BF16)
        return tc_field_bwd(d_raw, reinterpret_cast<const char*>(packed) + packed_layout().bf16_off, grads, d_enc_pos, d_enc_dir, ws, Q,
                            as_stream(stream));
    return fp32_mlp_bwd(d_raw, packed, grads, d_enc_pos, d_enc_dir, ws, Q, as_stream(stream));
}

extern "C" int nsb_field_bwd(const float* d_raw, const void* packed, float* grads, void* ws, size_t ws_bytes, int64_t Q,
                             int mode, void* stream) {
    if (Q != 0 && !grads) return NSB_E_BADARG;
    return nsb_field_bwd_ex(d_raw, packed, grads, nullptr, nullptr, ws, ws_bytes, Q, mode, stream);
}

// test hook (not part of include/nsb.h): tensor-core forward + fp32 dump of one layer's activations [Q,256]
extern "C" int nsb_debug_tc_layer(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm,
                                  const float* viewdirs, const void* packed, float* raw, float* dbg, int layer, int64_t B,
                                  int N, void* stream) {
    return tc_debug_layer(rays_o, rays_d, z, ray_norm, viewdirs, reinterpret_cast<const char*>(packed) + packed_layout().bf16_off,
                          raw, dbg, layer, B, N, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------------
// whole train step
// ---------------------------------------------------------------------------------------------------
namespace {
// one side stream (+ fork/join events) per device, created on first use; NSB_SIDE_STREAM=0 keeps everything on the caller's stream
struct SideStream { cudaStream_t stream; cudaEvent_t fork, join; };
SideStream* side_stream() {
    static SideStream table[64];
    static int state[64];          // 0 = not tried, 1 = ready, -1 = unavailable
    static const bool enabled = [] { const char* e = getenv("NSB_SIDE_STREAM"); return !(e && e[0] == '0'); }();
    static std::mutex init_mutex;  // first use from two host threads (one per device) must not race on the table
    int dev = 0;
    if (!enabled || cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(init_mutex);
    if (state[dev] == 0) {
        SideStream& s = table[dev];
        state[dev] = (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess &&
                      cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess &&
                      cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess) ? 1 : -1;
    }
    return state[dev] == 1 ? &table[dev] : nullptr;
}
struct TrainWs {
    float *zc, *w_c, *z_all, *raw_c, *raw_f, *d_raw, *d_raw_c, *comp_c, *comp_f, *g_c, *g_f;
    void *field_c, *field_f;
    size_t field_c_bytes, field_f_bytes, bytes;
    // ray gradients only (after everything above, so the layout without them is unchanged): encoding gradients of both passes
    // (63 + 27 floats per point each: 360 B per point in all) and the coarse pass's d rays_o / rays_d / viewdirs [3][B,3]
    float *d_ep_c, *d_ed_c, *d_ep_f, *d_ed_f, *d_rays_c;
};
TrainWs carve_train(void* base, int64_t B, int Nc, int Nf, int mode, bool ray_grads) {
    TrainWs t;
    char* p = reinterpret_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = p + off; off += align_up(bytes, 256); return r; };
    const int64_t Qc = B * (int64_t)Nc, Qf = B * (int64_t)(Nc + Nf);
    t.zc = (float*)take(Qc * 4); t.w_c = (float*)take(Qc * 4); t.z_all = (float*)take(Qf * 4);
    t.raw_c = (float*)take(Qc * 16); t.raw_f = (float*)take(Qf * 16); t.d_raw = (float*)take(Qf * 16); t.d_raw_c = (float*)take(Qc * 16);
    t.comp_c = (float*)take(B * 12); t.comp_f = (float*)take(B * 12); t.g_c = (float*)take(B * 12); t.g_f = (float*)take(B * 12);
    t.field_c_bytes = field_ws(Qc, mode, 1); t.field_f_bytes = field_ws(Qf, mode, 1);
    t.field_c = take(t.field_c_bytes); t.field_f = take(t.field_f_bytes);
    t.d_ep_c = t.d_ed_c = t.d_ep_f = t.d_ed_f = t.d_rays_c = nullptr;
    if (ray_grads) {
        t.d_ep_c = (float*)take(Qc * 63 * 4); t.d_ed_c = (float*)take(Qc * 27 * 4);
        t.d_ep_f = (float*)take(Qf * 63 * 4); t.d_ed_f = (float*)take(Qf * 27 * 4);
        t.d_rays_c = (float*)take(B * 36);
    }
    t.bytes = off;
    return t;
}
// fine-pass ray gradients += the coarse pass's, in that order (after the join of the two backward chains)
__global__ void add_coarse_ray_grads_kernel(float* __restrict__ d_o, float* __restrict__ d_d, float* __restrict__ d_v,
                                            const float* __restrict__ coarse, int64_t n3) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n3; i += (int64_t)gridDim.x * blockDim.x) {
        if (d_o) d_o[i] += coarse[i];
        if (d_d) d_d[i] += coarse[n3 + i];
        if (d_v) d_v[i] += coarse[2 * n3 + i];
    }
}
}  // namespace

extern "C" size_t nsb_train_workspace_bytes(int64_t B, int Nc, int Nf, int mode) {
    return carve_train(nullptr, B, Nc, Nf, mode, false).bytes;
}
extern "C" size_t nsb_train_workspace_bytes_ex(int64_t B, int Nc, int Nf, int mode, int ray_grads) {
    return carve_train(nullptr, B, Nc, Nf, mode, ray_grads != 0).bytes;
}

extern "C" int nsb_train_fwd_bwd_ex(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                                    const float* target, const void* packed_c, const void* packed_f, float* grads_c,
                                    float* grads_f, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes,
                                    int64_t B, int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags,
                                    int det_fine, int mode, float grad_scale, uint64_t seed, uint64_t step, const float* U,
                                    const float* u_fine, const float* noise_c, const float* noise_f, float* d_rays_o,
                                    float* d_rays_d, float* d_viewdirs, void* stream) {
    const bool ray_grads = d_rays_o || d_rays_d || d_viewdirs;
    if (!rays_o || !rays_d || !target || !packed_c || !packed_f || !scalars || !ws) return NSB_E_BADARG;
    // both gradient buffers, or neither (a frozen field: then only the ray gradients are computed)
    if (!grads_c != !grads_f || (!grads_c && !ray_grads) || (d_viewdirs && !viewdirs)) return NSB_E_BADARG;
    if (B < 1 || Nc < 2 || Nf < 1) return NSB_E_BADARG;
    TrainWs t = carve_train(ws, B, Nc, Nf, mode, ray_grads);
    if (ws_bytes < t.bytes) return NSB_E_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    const int Nt = Nc + Nf;
    const int64_t Qc = B * (int64_t)Nc, Qf = B * (int64_t)Nt;
    const uint32_t f = flags | NSB_TRAINING;
    // independent Philox streams per (step, purpose)
    const uint64_t s_jit = step * 8 + 0, s_u = step * 8 + 1, s_nc = step * 8 + 2, s_nf = step * 8 + 3;
    if (grads_c && grads_f == grads_c + NSB_N_PARAMS) {     // one flat buffer (the trainer's layout): one memset
        if (cudaMemsetAsync(grads_c, 0, 2 * sizeof(float) * NSB_N_PARAMS, st) != cudaSuccess) return NSB_E_CUDA;
    } else if (grads_c) {
        if (cudaMemsetAsync(grads_c, 0, sizeof(float) * NSB_N_PARAMS, st) != cudaSuccess) return NSB_E_CUDA;
        if (cudaMemsetAsync(grads_f, 0, sizeof(float) * NSB_N_PARAMS, st) != cudaSuccess) return NSB_E_CUDA;
    }
    // Forward chain (coarse pass, resampling, fine pass) of rays [b0, b0 + nb) on `strm`; Philox streams shifted by `sid`.
    // A half batch writes its own rows / tiles of every buffer, so the backward can treat the batch as a whole.
    auto forward = [&](int64_t b0, int64_t nb, uint64_t sid, void* strm) -> int {
        const float* rn = ray_norm ? ray_norm + b0 : nullptr;
        const float* vd = viewdirs ? viewdirs + 3 * b0 : nullptr;
        auto opt = [](const float* p, int64_t ofs) { return p ? p + ofs : nullptr; };
        float* zc = t.zc + b0 * Nc; float* z_all = t.z_all + b0 * Nt; float* w_c = t.w_c + b0 * Nc;
        float* raw_c = t.raw_c + 4 * b0 * Nc; float* raw_f = t.raw_f + 4 * b0 * Nt;
        // field workspaces: tile k of the stash lives k tiles in, and a half batch starts on a tile boundary (checked below)
        const size_t tile = mode == NSB_MODE_BF16 ? tc_stash_tile_bytes() : 0;
        const size_t off_c = (size_t)(b0 * Nc / 128) * tile, off_f = (size_t)(b0 * Nt / 128) * tile;
        NSB_TRY(nsb_stratified_z(zc, opt(U, b0 * Nc), nb, Nc, near_, far_, 1, seed, s_jit + sid, strm));                     // trainer.py:901-908
        NSB_TRY(nsb_field_fwd_rays(rays_o + 3 * b0, rays_d + 3 * b0, zc, rn, vd, packed_c, raw_c, static_cast<char*>(t.field_c) + off_c,
                                   t.field_c_bytes - off_c, nb, Nc, mode, 1, strm));
        // (sigma-noise draws are indexed by the sample's position in the WHOLE batch: the backward regenerates them in one launch)
        NSB_TRY(composite_raw_fwd_at(raw_c, opt(noise_c, b0 * Nc), noise_std, zc, rn, t.comp_c + 3 * b0, w_c, nullptr, nullptr, nb, Nc, f,
                                     seed, s_nc, b0 * Nc, strm));                                                            // :911-923
        NSB_TRY(nsb_resample_merge(zc, w_c, opt(u_fine, b0 * Nf), z_all, nullptr, nb, Nc, Nf, det_fine, seed, s_u + sid, strm));   // :926-934, :981
        NSB_TRY(nsb_field_fwd_rays(rays_o + 3 * b0, rays_d + 3 * b0, z_all, rn, vd, packed_f, raw_f, static_cast<char*>(t.field_f) + off_f,
                                   t.field_f_bytes - off_f, nb, Nt, mode, 1, strm));
        return composite_raw_fwd_at(raw_f, opt(noise_f, b0 * Nt), noise_std, z_all, rn, t.comp_f + 3 * b0, nullptr, nullptr, nullptr, nb, Nt,
                                    f, seed, s_nf, b0 * Nt, strm);                                                           // :984-996
    };
    // d raw of the whole batch straight from the target: the MSE gradient (:999-1004) is formed inside the compositor's backward
    // from the composite it recomputes anyway, so the loss kernel (scalars only) is off the critical path
    const float loss_scale = 2.0f * grad_scale / (3.0f * (float)B);
    auto composite_bwd = [&](bool fine, void* strm) -> int {
        if (fine)
            return nsb_composite_raw_bwd_mse(t.raw_f, noise_f, noise_std, t.z_all, ray_norm, target, loss_scale, t.d_raw, B, Nt, f, seed, s_nf, strm);
        return nsb_composite_raw_bwd_mse(t.raw_c, noise_c, noise_std, t.zc, ray_norm, target, loss_scale, t.d_raw_c, B, Nc, f, seed, s_nc, strm);
    };
    // Two half batches on two streams (tensor-core mode): each persistent field kernel ends with a partly filled round of
    // tiles (e.g. 768 tile pairs on 148 SMs = 5.19 rounds); with the other half's kernels in flight those SMs are not idle.
    SideStream* side = side_stream();
    const int64_t hb = B / 2;
    const bool split = side && mode == NSB_MODE_BF16 && B % 2 == 0 && hb >= 128 && (hb * Nc) % 128 == 0 && (hb * Nt) % 128 == 0;
    const uint64_t sid1 = 1ull << 40;                     // Philox stream shift of the second half
    void* sstream = side ? static_cast<void*>(side->stream) : stream;
    auto fork = [&]() { return cudaEventRecord(side->fork, st) == cudaSuccess && cudaStreamWaitEvent(side->stream, side->fork, 0) == cudaSuccess; };
    auto join = [&]() { return cudaEventRecord(side->join, side->stream) == cudaSuccess && cudaStreamWaitEvent(st, side->join, 0) == cudaSuccess; };
    if (split) {
        if (!fork()) return NSB_E_CUDA;
        NSB_TRY(forward(0, hb, 0, stream));
        NSB_TRY(forward(hb, hb, sid1, sstream));
        if (!join()) return NSB_E_CUDA;
    } else {
        NSB_TRY(forward(0, B, 0, stream));
    }
    // loss (:999-1006) and backward (:717).  The two backward chains are independent (coarse weights only feed the detached
    // resampling), so the coarse one runs on the side stream forked here and joined below: its CTAs fill the SMs the fine kernels
    // leave idle in their last round.  The loss scalars are computed at the head of the side stream.  Fork/join through events,
    // so the sequence stays graph-capturable.
    if (side && !fork()) return NSB_E_CUDA;
    // With ray gradients each pass's field backward also writes its encoding gradients, which nsb_encode_bwd_rays reduces to the
    // rays: the fine pass's straight into the outputs, the coarse pass's (side stream) into a buffer added after the join.
    NSB_TRY(composite_bwd(true, stream));
    NSB_TRY(nsb_field_bwd_ex(t.d_raw, packed_f, grads_f, t.d_ep_f, t.d_ed_f, t.field_f, t.field_f_bytes, Qf, mode, stream));
    if (ray_grads)
        NSB_TRY(nsb_encode_bwd_rays(t.d_ep_f, t.d_ed_f, rays_o, rays_d, t.z_all, ray_norm, viewdirs, d_rays_o, d_rays_d, d_viewdirs,
                                    B, Nt, stream));
    NSB_TRY(nsb_mse_loss(t.comp_c, t.comp_f, target, nullptr, nullptr, scalars, B, grad_scale, sstream));
    NSB_TRY(composite_bwd(false, sstream));
    NSB_TRY(nsb_field_bwd_ex(t.d_raw_c, packed_c, grads_c, t.d_ep_c, t.d_ed_c, t.field_c, t.field_c_bytes, Qc, mode, sstream));
    float* dr_c = t.d_rays_c;
    if (ray_grads)
        NSB_TRY(nsb_encode_bwd_rays(t.d_ep_c, t.d_ed_c, rays_o, rays_d, t.zc, ray_norm, viewdirs, d_rays_o ? dr_c : nullptr,
                                    d_rays_d ? dr_c + 3 * B : nullptr, d_viewdirs ? dr_c + 6 * B : nullptr, B, Nc, sstream));
    if (side && !join()) return NSB_E_CUDA;
    if (ray_grads) {
        const int64_t want = cdiv(3 * B, 256), cap = (int64_t)num_sms() * 8;
        add_coarse_ray_grads_kernel<<<(int)(want < cap ? want : cap), 256, 0, st>>>(d_rays_o, d_rays_d, d_viewdirs, dr_c, 3 * B);
        NSB_LAUNCH_CHECK("add_coarse_ray_grads_kernel");
    }
    if (comp_c && cudaMemcpyAsync(comp_c, t.comp_c, B * 12, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return NSB_E_CUDA;
    if (comp_f && cudaMemcpyAsync(comp_f, t.comp_f, B * 12, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return NSB_E_CUDA;
    return NSB_OK;
}

extern "C" int nsb_train_fwd_bwd(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                                 const float* target, const void* packed_c, const void* packed_f, float* grads_c,
                                 float* grads_f, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes,
                                 int64_t B, int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags,
                                 int det_fine, int mode, float grad_scale, uint64_t seed, uint64_t step, const float* U,
                                 const float* u_fine, const float* noise_c, const float* noise_f, void* stream) {
    if (!grads_c || !grads_f) return NSB_E_BADARG;
    return nsb_train_fwd_bwd_ex(rays_o, rays_d, ray_norm, viewdirs, target, packed_c, packed_f, grads_c, grads_f, scalars, comp_c, comp_f,
                                ws, ws_bytes, B, Nc, Nf, near_, far_, noise_std, flags, det_fine, mode, grad_scale, seed, step, U, u_fine,
                                noise_c, noise_f, nullptr, nullptr, nullptr, stream);
}

// ---------------------------------------------------------------------------------------------------
// whole optimisation step, replayable as a CUDA graph
// ---------------------------------------------------------------------------------------------------
namespace nsb {
int adam_impl(float* params, const float* grads, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps, int64_t t,
              float grad_scale, const uint64_t* t_dev, float eta_min, int64_t T_max, const float* loss_guard, void* stream);
int adam_allreduce_impl(float* const* params, float* const* m, float* const* v, int n_nets, const void* const* peer_grads,
                        void* const* peer_flags, int rank, int world, uint32_t epoch, int64_t n, float lr, float beta1,
                        float beta2, float eps, int64_t t, float grad_scale, const uint64_t* t_dev, float eta_min, int64_t T_max,
                        const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync, const float* loss_guard, void* stream);
__global__ void counter_inc_kernel(uint64_t* c) { if (threadIdx.x == 0 && blockIdx.x == 0) *c += 1; }
}  // namespace nsb

extern "C" int nsb_train_step(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                              const float* target, float* const* params, float* const* m, float* const* v, void* const* packed,
                              float* grads, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes, int64_t B,
                              int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags, int det_fine, int mode,
                              uint64_t seed, float lr, float lr_eta_min, int64_t lr_T_max, float beta1, float beta2, float eps,
                              float grad_clip_norm, uint64_t* step_counter,
                              const void* const* peer_grads, const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync,
                              void* const* peer_flags, int rank, int world, void* stream) {
    if (!params || !m || !v || !packed || !grads || !step_counter) return NSB_E_BADARG;
    for (int k = 0; k < 2; ++k)
        if (!params[k] || !m[k] || !v[k] || !packed[k]) return NSB_E_BADARG;
    if (world < 1 || (world > 1 && (!peer_grads || !peer_flags))) return NSB_E_BADARG;
    // clipping needs the norm of the REDUCED gradient before any parameter moves: not available inside the fused exchange
    if (grad_clip_norm > 0.f && world > 1) return NSB_E_BADARG;
    // forward + backward with the Philox streams shifted by the device-side step count
    g_step_dev = step_counter;
    int rc = nsb_train_fwd_bwd(rays_o, rays_d, ray_norm, viewdirs, target, packed[0], packed[1], grads, grads + NSB_N_PARAMS, scalars,
                               comp_c, comp_f, ws, ws_bytes, B, Nc, Nf, near_, far_, noise_std, flags, det_fine, mode, 1.0f, seed,
                               /*step=*/0, nullptr, nullptr, nullptr, nullptr, stream);
    g_step_dev = nullptr;
    if (rc) return rc;
    // optimiser (+ gradient exchange over peer memory), t = *step_counter + 1
    if (world > 1) {
        NSB_TRY(adam_allreduce_impl(params, m, v, 2, peer_grads, peer_flags, rank, world, 0, NSB_N_PARAMS, lr, beta1, beta2, eps, 1,
                                    1.0f / (float)world, step_counter, lr_eta_min, lr_T_max, mc_grads, mc_reduced, reduced, local_sync, scalars, stream));
    } else {        // one rank: the same kernel without the exchange -- both nets in one launch
        if (grad_clip_norm > 0.f)      // trainer.py:719-721; scratch = scalars[4]
            NSB_TRY(nsb_grad_clip(grads, 2 * (int64_t)NSB_N_PARAMS, grad_clip_norm, 1.0f, scalars + 4, stream));
        const void* own[1] = {grads};
        NSB_TRY(adam_allreduce_impl(params, m, v, 2, own, nullptr, 0, 1, 0, NSB_N_PARAMS, lr, beta1, beta2, eps, 1, 1.0f, step_counter,
                                    lr_eta_min, lr_T_max, nullptr, nullptr, nullptr, nullptr, scalars, stream));
    }
    const float* cparams[2] = {params[0], params[1]};
    g_pack_counter = mode == NSB_MODE_BF16 ? step_counter : nullptr;      // the tensor-core pack kernel increments it as its last act
    rc = nsb_pack_weights_batch(cparams, packed, 2, mode | NSB_PACK_TRAIN_ONLY, stream);           // inference images: on demand
    g_pack_counter = nullptr;
    if (rc) return rc;
    if (mode != NSB_MODE_BF16) {
        counter_inc_kernel<<<1, 32, 0, as_stream(stream)>>>(step_counter);
        NSB_LAUNCH_CHECK("counter_inc_kernel");
    }
    return NSB_OK;
}

// ---------------------------------------------------------------------------------------------------
// eval ray tile
// ---------------------------------------------------------------------------------------------------
namespace {
struct RenderWs {
    float *zc, *w_c, *z_all, *raw;
    void* field;
    size_t field_bytes, bytes;
};
RenderWs carve_render(void* base, int64_t B, int Nc, int Nf, int mode) {
    RenderWs t;
    char* p = reinterpret_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = p + off; off += align_up(bytes, 256); return r; };
    const int Nt = Nc + (Nf > 0 ? Nf : 0);
    t.zc = (float*)take(B * (int64_t)Nc * 4); t.w_c = (float*)take(B * (int64_t)Nc * 4);
    t.z_all = (float*)take(B * (int64_t)Nt * 4); t.raw = (float*)take(B * (int64_t)Nt * 16);
    t.field_bytes = field_ws(B * (int64_t)Nt, mode, 0);
    t.field = take(t.field_bytes);
    t.bytes = off;
    return t;
}
}  // namespace

extern "C" size_t nsb_render_workspace_bytes(int64_t B, int Nc, int Nf, int mode) {
    return carve_render(nullptr, B, Nc, Nf, mode).bytes;
}

extern "C" int nsb_render_rays(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                               const void* packed_c, const void* packed_f, float* rgb, float* acc, float* depth, void* ws,
                               size_t ws_bytes, int64_t B, int Nc, int Nf, float near_, float far_, uint32_t flags,
                               int mode, void* stream) {
    if (B == 0) return NSB_OK;
    if (!rays_o || !rays_d || !packed_c || !rgb || !ws || B < 0 || Nc < 1) return NSB_E_BADARG;
    const bool fine = Nf > 0 && packed_f != nullptr;                                                                   // render_utils.py:381
    if (fine && Nc < 2) return NSB_E_BADARG;
    RenderWs t = carve_render(ws, B, Nc, fine ? Nf : 0, mode);
    if (ws_bytes < t.bytes) return NSB_E_WORKSPACE;
    const uint32_t f = flags & ~NSB_TRAINING;
    NSB_TRY(nsb_stratified_z(t.zc, nullptr, B, Nc, near_, far_, 0, 0, 0, stream));                                      // :330-331,351
    NSB_TRY(nsb_field_fwd_rays(rays_o, rays_d, t.zc, ray_norm, viewdirs, packed_c, t.raw, t.field, t.field_bytes, B, Nc, mode, 0, stream));
    if (!fine)
        return nsb_composite_raw_fwd(t.raw, nullptr, 0.f, t.zc, ray_norm, rgb, nullptr, acc, depth, B, Nc, f, 0, 0, stream);
    NSB_TRY(nsb_composite_raw_fwd(t.raw, nullptr, 0.f, t.zc, ray_norm, rgb, t.w_c, nullptr, nullptr, B, Nc, f, 0, 0, stream));   // :362-375
    NSB_TRY(nsb_resample_merge(t.zc, t.w_c, nullptr, t.z_all, nullptr, B, Nc, Nf, 1, 0, 0, stream));                   // :388-395
    NSB_TRY(nsb_field_fwd_rays(rays_o, rays_d, t.z_all, ray_norm, viewdirs, packed_f, t.raw, t.field, t.field_bytes, B, Nc + Nf, mode, 0, stream));
    return nsb_composite_raw_fwd(t.raw, nullptr, 0.f, t.z_all, ray_norm, rgb, nullptr, acc, depth, B, Nc + Nf, f, 0, 0, stream);   // :399-417
}
