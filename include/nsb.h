/* nsb.h -- C ABI of libnsb.so, the B200 (sm_100a) engine for the vanilla-NeRF ray-march path of
 * evan-wes/nerf-sandbox.
 *
 * The reference has no FFI: its seam is a set of Python callables bound by name
 * (train/trainer.py:46-54, utils/render_utils.py:24-25, utils/validation_renderer.py:16-24).  Each
 * entry point below states which of those callables (file:line in the reference) it replaces.
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller (PyTorch) owns all
 *     memory including workspaces, so the caching allocator and CUDA-graph capture keep working;
 *   - fp32, contiguous, row-major; ray-major then sample-major: z[b*N+i], raw[(b*N+i)*4+c];
 *   - `stream` is a cudaStream_t passed as void*; no call synchronises or allocates;
 *   - return 0 on success, a negative NSB_E_* code otherwise (nsb_error_string explains it);
 *     the Python wrappers raise RuntimeError/ValueError like the reference does;
 *   - nullable arguments are marked [opt];
 *   - threading: the library keeps no state per call except (a) thread-local markers set for the duration of nsb_train_step
 *     and (b) ONE helper stream + event pair per device, created on first use, on which nsb_train_fwd_bwd(_ex) / nsb_train_step
 *     run half batches and the coarse backward chain.  Calls on different devices are independent; on one device, two host
 *     threads must not be inside nsb_train_fwd_bwd(_ex) / nsb_train_step at the same time (the reference is single-threaded,
 *     single-stream; NSB_SIDE_STREAM=0 removes the helper stream and with it this restriction).
 */
#ifndef NSB_H_
#define NSB_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSB_OK 0
#define NSB_E_BADARG (-1)     /* shape / flag the path does not support                         */
#define NSB_E_WORKSPACE (-2)  /* workspace too small (see nsb_field_workspace_bytes)            */
#define NSB_E_CUDA (-3)       /* a CUDA runtime call or launch failed; see nsb_last_cuda_error  */
#define NSB_E_ARCH (-4)       /* device is not sm_100 (every tcgen05 kernel: both modes' defaults) */

/* flags for the compositor / forward pass */
#define NSB_WHITE_BKGD 1u        /* render_utils.py:161-162 */
#define NSB_INFINITE_LAST_BIN 2u /* render_utils.py:132-135 */
#define NSB_TRAINING 4u          /* render_utils.py:239: add raw noise to sigma before the activation */
#define NSB_SIGMA_SOFTPLUS 8u    /* render_utils.py:243-246: sigma = softplus(raw) instead of relu(raw) (raw entry points) */

/* arithmetic mode of the field (encoder + MLP) kernels */
#define NSB_MODE_FP32 0  /* fp32 activations / gradients in HBM, the 1e-4 parity mode: layer GEMMs on tcgen05 with
                          * operands split into three bf16 terms (fp32-grade products) */
#define NSB_MODE_BF16 1  /* tcgen05 tensor cores, bf16 operands, fp32 accumulate in TMEM     */

/* NeRF(63,27,8,256,skip_pos=4) -- models/mlps.py:41-134.  Flat parameter order is the reference's
 * state_dict order: mlp.0.weight, mlp.0.bias, ..., mlp.7.*, feature.*, sigma_out.*, color_fc.*,
 * color_out.* (SURVEY.md section 5). */
#define NSB_N_PARAMS 595844

int nsb_version(void);
const char* nsb_error_string(int code);
const char* nsb_last_cuda_error(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
int64_t nsb_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * K2  samplers
 * ---------------------------------------------------------------------------------------------- */

/* Stratified coarse samples; replaces the inline code of Trainer._train_step, train/trainer.py:901-908
 * (jittered) and render_image_chunked, utils/render_utils.py:330-331,351 (U == NULL && !jitter: plain
 * linspace).  z[B,Nc].  U[B,Nc] [opt] explicit uniforms in [0,1) (parity tests); when NULL and jitter!=0
 * uniforms come from Philox(seed, offset). Bit-exact with the reference given the same U. */
int nsb_stratified_z(float* z, const float* U, int64_t B, int Nc, float near_, float far_, int jitter,
                     uint64_t seed, uint64_t offset, void* stream);

/* sample_pdf, utils/sampling_utils.py:5-64.  bins[B,bins_cols] with bins_cols == M (midpoints) or M+1
 * (edges); weights[B,M]; out[B,n].  u[B,n] [opt] explicit uniforms; cdf_in[B,M+1] [opt] replaces the
 * CDF built from weights (the bit-exact index test feeds the reference's CDF); inds_out[B,n] [opt]
 * receives searchsorted(cdf,u,right=True) as int64.  deterministic != 0: u = linspace(0,1,n). */
int nsb_sample_pdf(const float* bins, int bins_cols, const float* weights, int M, const float* u,
                   const float* cdf_in, float* out, int64_t* inds_out, int64_t B, int n, int deterministic,
                   uint64_t seed, uint64_t offset, void* stream);

/* Fused hierarchical resampling: interval weights (train/trainer.py:926-928) + sample_pdf (:930) +
 * sort(cat(zc,zf)) (:981).  zc[B,Nc] sorted, w_c[B,Nc]; z_all[B,Nc+Nf]; z_fine[B,Nf] [opt] unsorted
 * samples as sample_pdf returns them; u[B,Nf] [opt]. */
int nsb_resample_merge(const float* zc, const float* w_c, const float* u, float* z_all, float* z_fine,
                       int64_t B, int Nc, int Nf, int deterministic, uint64_t seed, uint64_t offset,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3  compositor
 * ---------------------------------------------------------------------------------------------- */

/* volume_render_rays, utils/render_utils.py:108-167.  rgb[B,N,3], sigma[B,N], z[B,N],
 * ray_norm[B] [opt]; comp[B,3], weights[B,N] [opt], acc[B], depth[B]. flags: NSB_WHITE_BKGD,
 * NSB_INFINITE_LAST_BIN. */
int nsb_composite_fwd(const float* rgb, const float* sigma, const float* z, const float* ray_norm,
                      float* comp, float* weights, float* acc, float* depth, int64_t B, int N,
                      uint32_t flags, float eps, void* stream);
/* autograd of the above w.r.t. (rgb, sigma).  g_comp[B,3]; g_weights[B,N], g_acc[B], g_depth[B] [opt].
 * d_rgb[B,N,3], d_sigma[B,N]. */
int nsb_composite_bwd(const float* rgb, const float* sigma, const float* z, const float* ray_norm,
                      const float* g_comp, const float* g_weights, const float* g_acc, const float* g_depth,
                      float* d_rgb, float* d_sigma, int64_t B, int N, uint32_t flags, float eps, void* stream);

/* Fused head activation + compositor: the tail of nerf_forward_pass, utils/render_utils.py:230-247
 * (sigmoid on rgb logits, sigma = relu(raw + noise*std) when NSB_TRAINING) followed by :269-276.
 * raw[B*N,4] = NeRF.forward output [r,g,b,sigma]; noise[B*N] [opt] explicit N(0,1) draws, else
 * Philox(seed, offset) when NSB_TRAINING and noise_std > 0. */
int nsb_composite_raw_fwd(const float* raw, const float* noise, float noise_std, const float* z,
                          const float* ray_norm, float* comp, float* weights, float* acc, float* depth,
                          int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset, void* stream);
int nsb_composite_raw_bwd(const float* raw, const float* noise, float noise_std, const float* z,
                          const float* ray_norm, const float* g_comp, float* d_raw, int64_t B, int N,
                          uint32_t flags, uint64_t seed, uint64_t offset, void* stream);
/* The same with the gradients of every output of volume_render_rays (render_utils.py:141-167): g_comp[B,3], g_weights[B,N],
 * g_acc[B], g_depth[B], each [opt] (a missing one counts as zero), at least one given -- a depth or opacity loss, or a loss on
 * the weights, reaches the field through d_raw.  nsb_composite_raw_bwd is this call with g_comp only.  No gradient w.r.t. z or
 * ray_norm. */
int nsb_composite_raw_bwd_ex(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm,
                             const float* g_comp, const float* g_weights, const float* g_acc, const float* g_depth, float* d_raw,
                             int64_t B, int N, uint32_t flags, uint64_t seed, uint64_t offset, void* stream);

/* nsb_composite_raw_bwd with the step's loss gradient formed in place (train/trainer.py:999-1004 + :717): instead of g_comp it
 * takes target[B,3] and loss_scale = 2 * grad_scale / (3 * B_total), and uses dL/dcomp = (guard(comp) - guard(target)) *
 * loss_scale on the composite it recomputes anyway (guard = nan_to_num(nan=0, posinf=1, neginf=0).clamp(0,1)) -- the MSE
 * kernel then only produces the scalars and is off the step's critical path. */
int nsb_composite_raw_bwd_mse(const float* raw, const float* noise, float noise_std, const float* z, const float* ray_norm,
                              const float* target, float loss_scale, float* d_raw, int64_t B, int N, uint32_t flags,
                              uint64_t seed, uint64_t offset, void* stream);

/* Loss of Trainer._train_step, train/trainer.py:999-1006: guards + mse(comp_c)+mse(comp_f) and its
 * gradient.  scalars[4] = {loss, psnr, mse_c, mse_f} (device).  g_c/g_f[B,3] = dloss/dcomp * grad_scale.
 * comp_c may be NULL (coarse-only). */
int nsb_mse_loss(const float* comp_c, const float* comp_f, const float* target, float* g_c, float* g_f,
                 float* scalars, int64_t B, float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1  field: positional encoder + 8x256 skip MLP
 * ---------------------------------------------------------------------------------------------- */

/* PositionalEncoder.forward, models/encoders.py:73-106.  x[Q,D] -> out[Q, D*(include_input + 2L)],
 * order [x | sin(2^k x_d) k-major | cos(...)]. */
int nsb_encode(const float* x, float* out, int64_t Q, int D, int L, int include_input, void* stream);
/* Its autograd (encoders.py:101-104 through torch's sin/cos backward): g_out[Q, D*(include_input + 2L)] -> g_x[Q,D] =
 * [include_input] g + sum_k 2^k (cos(2^k x) g_sin_k - sin(2^k x) g_cos_k). */
int nsb_encode_bwd(const float* x, const float* g_out, float* g_x, int64_t Q, int D, int L, int include_input, void* stream);
/* Backward of the points + encodings step of nerf_forward_pass (render_utils.py:211-223, gamma(x) with L = 10, gamma(d) with
 * L = 4, both with the input): d_enc_pos[B*N,63], d_enc_dir[B*N,27] -> d_rays_o[B,3] = sum over samples of d pts,
 * d_rays_d[B,3] = sum of d pts * (z * norm), and the view-direction term through F.normalize's backward (eps 1e-12) into
 * d_viewdirs[B,3], or into d_rays_d when viewdirs is NULL.  Outputs [opt], at least one.  Inputs as nsb_field_fwd_rays.
 * Sums run in a fixed order (no atomics): bitwise repeatable.  z and ray_norm get no gradient. */
int nsb_encode_bwd_rays(const float* d_enc_pos, const float* d_enc_dir, const float* rays_o, const float* rays_d, const float* z,
                        const float* ray_norm, const float* viewdirs, float* d_rays_o, float* d_rays_d, float* d_viewdirs,
                        int64_t B, int N, void* stream);

/* Packed weights of one NeRF: fp32 padded rows (heads and biases of the fp32 mode), and images in tcgen05 operand layout for the tensor
 * paths -- bf16 (training forward), transposed bf16 (dgrad), fp16 (inference forward) and the fp16 low halves of the
 * split used by the fp32-accurate inference forward, and bf16 term images (w = w0 + w1 + w2) of every weight matrix, plain
 * and transposed, for the fp32 mode's tensor-core layer GEMMs.  Sizes in bytes. */
size_t nsb_packed_weights_bytes(void);
/* params: flat fp32 [NSB_N_PARAMS] in state_dict order -> packed (call after every optimiser step).
 * mode selects which section is refreshed: NSB_MODE_FP32, NSB_MODE_BF16, or -1 for both; OR-ing NSB_PACK_TRAIN_ONLY into it
 * skips the two inference-only fp16 images (what a training loop does between evaluations: re-pack fully before the next
 * inference call). */
#define NSB_PACK_TRAIN_ONLY 0x100
int nsb_pack_weights(const float* params, void* packed, int mode, void* stream);

/* The same for up to four nets in one call (training re-packs coarse + fine after every optimiser step: one kernel launch in
 * tensor-core mode).  params / packed: HOST arrays of n_nets device pointers. */
int nsb_pack_weights_batch(const float* const* params, void* const* packed, int n_nets, int mode, void* stream);

/* Workspace for one pass over Q = B*N points.  stash != 0 keeps what the backward needs. */
size_t nsb_field_workspace_bytes(int64_t Q, int mode, int stash);

/* NeRF.forward, models/mlps.py:192-278, on materialised encodings: enc_pos[Q,63], enc_dir[Q,27] ->
 * raw[Q,4].  (The module-level drop-in; the fused entry below never materialises the encodings.) */
int nsb_field_fwd_enc(const float* enc_pos, const float* enc_dir, const void* packed, float* raw,
                      void* ws, size_t ws_bytes, int64_t Q, int mode, int stash, void* stream);

/* Points + encodings + MLP of nerf_forward_pass, utils/render_utils.py:211-261: pts = o + d*(z*norm),
 * viewdirs normalised (:219) and broadcast per sample, gamma(x), gamma(d), NeRF.forward.
 * rays_o[B,3], rays_d[B,3], z[B,N], ray_norm[B] [opt], viewdirs[B,3] [opt: falls back to rays_d]. */
int nsb_field_fwd_rays(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm,
                       const float* viewdirs, const void* packed, float* raw, void* ws, size_t ws_bytes,
                       int64_t B, int N, int mode, int stash, void* stream);

/* Parameter gradients of the pass whose activations are stashed in ws: grads[NSB_N_PARAMS] (flat,
 * state_dict order) += dL/dparams given d_raw[Q,4].  (nsb_field_bwd_ex with no input gradients.) */
int nsb_field_bwd(const float* d_raw, const void* packed, float* grads, void* ws, size_t ws_bytes,
                  int64_t Q, int mode, void* stream);
/* NeRF.forward's autograd w.r.t. its parameters AND its inputs (mlps.py:221-278): grads [opt] as above, d_enc_pos[Q,63] [opt] and
 * d_enc_dir[Q,27] [opt] are overwritten with dL/d gamma(x) = dY_0 W_0[:, 0:63] + dY_4 W_4[:, 256:319] (layer 4's input is
 * [h, gamma(x)], mlps.py:224-227) and dL/d gamma(d) = dY_9 W_cfc[:, 256:283] (dY_l = gradient of layer l's pre-activation).
 * At least one output.  grads == NULL is a frozen field: no weight-gradient kernel runs at all. */
int nsb_field_bwd_ex(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws,
                     size_t ws_bytes, int64_t Q, int mode, void* stream);

/* torch.optim.Adam step (train/trainer.py:383-386, :722) on flat buffers; grads are multiplied by
 * grad_scale first (1/world_size after a sum-allreduce). t is the 1-based step count.
 * loss_guard [opt]: device pointer to the step's loss; when it is not finite the update is skipped, as the reference
 * loop does (train/trainer.py:713-716). */
int nsb_adam_step(float* params, const float* grads, float* m, float* v, int64_t n, float lr, float beta1,
                  float beta2, float eps, int64_t t, float grad_scale, const float* loss_guard, void* stream);

/* torch.nn.utils.clip_grad_norm_(params, max_norm) (train/trainer.py:719-721) on a flat gradient buffer: the total L2 norm
 * of pre_scale * grads[n] is taken over ALL n entries (both nets when they share one buffer) and grads *= min(1,
 * max_norm / (norm + 1e-6)).  pre_scale = the grad_scale the following Adam call will apply (1/world after a sum-allreduce).
 * scratch: one float of device memory. */
int nsb_grad_clip(float* grads, int64_t n, float max_norm, float pre_scale, float* scratch, void* stream);

/* Data-parallel tail of a step in ONE kernel (SURVEY 8e; replaces `all_reduce(grads)` + Adam, train/trainer.py:717-725 under
 * DDP): waits until every rank's gradient buffer of this epoch is complete (flag exchange through peer memory), sums the
 * `world` buffers in rank order with loads that go to the peers' HBM over NVLink/NVSwitch, and applies Adam (grads times
 * grad_scale) to this rank's full parameter copies; the replicas stay bit-identical.
 * params / m / v: HOST arrays of n_nets device pointers, n floats each (one entry per net); net k's gradients are
 * peer_grads[r] + k * n.  peer_grads[r] / peer_flags[r] (HOST arrays of `world` device addresses valid in this process:
 * symmetric / peer-mapped allocations): rank r's gradient buffer [n_nets * n] and flag block (uint32[3 * world], zeroed once: epoch flags, then one "my loss is
 * not finite" word per rank and epoch parity).
 * `epoch` starts at 1 and increases by one per step on every rank; the caller alternates between two gradient buffers by
 * epoch parity (that is what makes one flag exchange per step sufficient).  n % 4 == 0.
 * mc_grads (optional): multicast (NVLS) address of the same gradient buffers; when given, the sum is one
 * `multimem.ld_reduce` per 16 bytes -- the NVSwitch reduces, every rank receives n_nets * n floats instead of world times that.
 * mc_reduced / reduced / local_sync (optional, all three or none; need mc_grads): the TWO-PHASE exchange for 4+ ranks.  With
 * mc_grads alone every rank pulls the whole reduced buffer, i.e. every GPU's buffer is read `world` times by the switch;
 * here rank r reduces only its 1/world slice and multicast-stores it (`multimem.st`) into every rank's reduced-gradient
 * buffer -- mc_reduced = multicast address, reduced = this rank's own copy, both n_nets * n floats of symmetric memory --,
 * a second flag round follows, and Adam runs on the local copy (two launches).  local_sync: 4 device ints of this rank,
 * zeroed once.  The flag blocks then hold uint32[4 * world].
 * loss_guard [opt]: this rank's loss (device); a non-finite loss on ANY rank makes EVERY rank skip the update
 * (train/trainer.py:713-716, made collective so the replicas stay identical). */
int nsb_adam_allreduce_step(float* const* params, float* const* m, float* const* v, int n_nets, const void* const* peer_grads,
                            const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync,
                            void* const* peer_flags, int rank, int world, uint32_t epoch, int64_t n, float lr,
                            float beta1, float beta2, float eps, int64_t t, float grad_scale, const float* loss_guard, void* stream);

/* Health of the peer-memory exchange above.  A rank waits NSB_PEER_TIMEOUT_S seconds (environment, default 600 -- a peer
 * may be validating, checkpointing or stalled on data) for its peers' flags; when that expires the kernel skips the update,
 * records the peer it was waiting for and returns normally (no trap: the CUDA context stays usable).  *code = 0 when every
 * exchange so far completed, else 1 + the rank that never arrived.  Synchronises the device (a 4-byte read-back); the
 * trainer calls it whenever it reads the step's scalars on the host.  No counterpart in the reference (single GPU). */
int nsb_peer_status(int* code);

/* ------------------------------------------------------------------------------------------------
 * Whole-path entry points (one host call per step / per ray tile)
 * ---------------------------------------------------------------------------------------------- */

size_t nsb_train_workspace_bytes(int64_t B, int Nc, int Nf, int mode);

/* One whole optimisation step -- nsb_train_fwd_bwd, Adam on both nets (with the gradient exchange over peer memory when
 * world > 1, see nsb_adam_allreduce_step) and the re-pack -- with the STEP COUNT IN DEVICE MEMORY, so the launch sequence
 * can be captured once into a CUDA graph and replayed (train/trainer.py:702-729 without per-step host work): Philox streams
 * use step = *step_counter, Adam and the flag epoch use t = *step_counter + 1, and the last kernel increments the counter.
 * params / m / v / packed: HOST arrays of two device pointers (coarse, fine); grads: [2 * NSB_N_PARAMS] (with world > 1 this
 * rank's buffer of the current epoch parity, i.e. capture one graph per parity); draws are always generated in-kernel.
 * lr_T_max > 0: the learning rate follows CosineAnnealingLR(T_max, eta_min) from base `lr` (make_scheduler, train/trainer.py:81-88),
 * evaluated on the device from the step count; lr_T_max <= 0: constant lr.
 * scalars[8]: {loss, psnr, mse_c, mse_f, squared gradient norm (when clipping), 3 spare}.  A non-finite loss skips the
 * optimiser update (train/trainer.py:713-716; the counter still advances).  grad_clip_norm > 0: clip_grad_norm_ over both
 * nets before Adam (:719-721) -- single rank only (world > 1 returns NSB_E_BADARG: the norm of the reduced gradient is not
 * available inside the fused exchange; use the NCCL path + nsb_grad_clip). */
int nsb_train_step(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                   const float* target, float* const* params, float* const* m, float* const* v, void* const* packed,
                   float* grads, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes, int64_t B,
                   int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags, int det_fine, int mode,
                   uint64_t seed, float lr, float lr_eta_min, int64_t lr_T_max, float beta1, float beta2, float eps,
                   float grad_clip_norm, uint64_t* step_counter,
                   const void* const* peer_grads, const void* mc_grads, void* mc_reduced, const float* reduced, int* local_sync,
                   void* const* peer_flags, int rank, int world, void* stream);

/* Trainer._train_step + loss.backward(), train/trainer.py:876-1013 and :717.  Batch tensors as
 * trainer.py:880-884.  grads_c/grads_f[NSB_N_PARAMS] are overwritten with dloss/dparams * grad_scale.
 * Explicit random draws [opt]: U[B,Nc], u_fine[B,Nf], noise_c[B*Nc], noise_f[B*(Nc+Nf)].
 * scalars[4] = {loss, psnr, mse_c, mse_f}; comp_c/comp_f[B,3] [opt]. */
int nsb_train_fwd_bwd(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                      const float* target, const void* packed_c, const void* packed_f, float* grads_c,
                      float* grads_f, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes,
                      int64_t B, int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags,
                      int det_fine, int mode, float grad_scale, uint64_t seed, uint64_t step, const float* U,
                      const float* u_fine, const float* noise_c, const float* noise_f, void* stream);

/* Workspace of nsb_train_fwd_bwd_ex: with ray_grads != 0 it holds the encoding gradients of both passes as well, 360 B more per
 * point (B * (2 Nc + Nf) points).  ray_grads == 0 is nsb_train_workspace_bytes. */
size_t nsb_train_workspace_bytes_ex(int64_t B, int Nc, int Nf, int mode, int ray_grads);

/* nsb_train_fwd_bwd that also returns the gradient of the step's loss (times grad_scale) w.r.t. its rays -- what autograd gives
 * rays_o, rays_d and viewdirs in the reference's _train_step: d_rays_o[B,3], d_rays_d[B,3], d_viewdirs[B,3], each [opt] and
 * overwritten, each the sum of the coarse and the fine pass (fine first, then coarse, in a fixed order: bitwise repeatable).
 * d_viewdirs needs viewdirs; without viewdirs the view-direction term goes to d_rays_d.  grads_c / grads_f: both or neither;
 * neither (with a ray output) is a frozen field, and no weight-gradient kernel runs.  z and ray_norm get no gradient, so for
 * NDC rays, whose marching norm depends on the pose, a pose gradient built on these is incomplete.  Workspace:
 * nsb_train_workspace_bytes_ex(..., ray_grads = 1) when a ray output is given.  With no ray output this is nsb_train_fwd_bwd:
 * the same launches in the same order. */
int nsb_train_fwd_bwd_ex(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                         const float* target, const void* packed_c, const void* packed_f, float* grads_c,
                         float* grads_f, float* scalars, float* comp_c, float* comp_f, void* ws, size_t ws_bytes,
                         int64_t B, int Nc, int Nf, float near_, float far_, float noise_std, uint32_t flags,
                         int det_fine, int mode, float grad_scale, uint64_t seed, uint64_t step, const float* U,
                         const float* u_fine, const float* noise_c, const float* noise_f, float* d_rays_o,
                         float* d_rays_d, float* d_viewdirs, void* stream);

size_t nsb_render_workspace_bytes(int64_t B, int Nc, int Nf, int mode);

/* One ray tile of render_image_chunked, utils/render_utils.py:337-417 (perturb=False): coarse linspace,
 * coarse pass, interval weights + deterministic sample_pdf + merge, fine pass.  Nf <= 0 or packed_f ==
 * NULL: coarse only (:381-385).  rgb[B,3], acc[B], depth[B]. */
int nsb_render_rays(const float* rays_o, const float* rays_d, const float* ray_norm, const float* viewdirs,
                    const void* packed_c, const void* packed_f, float* rgb, float* acc, float* depth, void* ws,
                    size_t ws_bytes, int64_t B, int Nc, int Nf, float near_, float far_, uint32_t flags, int mode,
                    void* stream);

/* ------------------------------------------------------------------------------------------------
 * Ray generation (the producer of the path's inputs; SURVEY section 8f rank 1)
 * ---------------------------------------------------------------------------------------------- */

/* get_camera_rays, utils/ray_utils.py:10-136.  K_host[9] (3x3 row-major) and c2w_host[3 x c2w_cols]
 * (c2w_cols must be 4; rows of a (3,4) or (4,4) pose) are HOST pointers.  convention: 0 opengl/blender/nerf,
 * 1 opencv/colmap, 2 pytorch3d (:69-77).  pixels_xy[n_pixels,2] [opt, device] selects pixels (x,y), otherwise
 * the full H*W row-major grid.  Outputs (device): o_world[n,3], d_world_unit[n,3], d_world_norm[n],
 * o_march[n,3], d_march_unit[n,3], d_march_norm[n] -- the reference's 6-tuple; as_ndc applies the NDC
 * warp of :92-126 to the marching rays. */
int nsb_camera_rays(int H, int W, const float* K_host, const float* c2w_host, int c2w_cols, int convention,
                    int pixel_center, int as_ndc, float near_plane, const float* pixels_xy, int64_t n_pixels,
                    float* o_world, float* d_world_unit, float* d_world_norm, float* o_march, float* d_march_unit,
                    float* d_march_norm, void* stream);

/* Backward of nsb_camera_rays / nsb_sample_pixel_batch w.r.t. the poses (iNeRF / BARF-style pose refinement): the exact adjoint
 * of the six outputs in world and NDC mode.  Ks[F,4] = (fx,fy,cx,cy) and c2ws[F,12] (row-major 3x4) are DEVICE arrays, as for
 * the sampler; fids[n] [opt] is each ray's frame (NULL: every ray is frame 0; an id outside [0,F) contributes nothing) and
 * pixels_xy[n,2] [opt] its pixel (NULL: the full row-major H*W grid, and then n must be H*W) -- what the sampler returns.
 * Upstream gradients g_*[n,3] / g_*_norm[n], each [opt] (a missing one counts as zero), at least one given.
 * d_c2ws[F,12] is overwritten with dL/dc2w[:3,:4]; a frame no ray belongs to gets exactly zero.  The per-frame sums use no
 * atomics (block partials in ws, then a second pass in block order): bitwise repeatable.  ws: at least
 * nsb_camera_rays_bwd_workspace_bytes(n, F) bytes.  Two launches. */
size_t nsb_camera_rays_bwd_workspace_bytes(int64_t n, int F);
int nsb_camera_rays_bwd(int H, int W, const float* Ks, const float* c2ws, int F, const int* fids, int convention,
                        int pixel_center, int as_ndc, float near_plane, const float* pixels_xy, int64_t n,
                        const float* g_o_world, const float* g_d_world_unit, const float* g_d_world_norm,
                        const float* g_o_march, const float* g_d_march_unit, const float* g_d_march_norm,
                        float* d_c2ws, void* ws, size_t ws_bytes, void* stream);

/* Device-side pixel/ray batch sampler (SURVEY section 8f rank 2): RandomPixelRaySampler.__iter__,
 * data/samplers.py:134-290, with the images resident in HBM and no host round trip.  images[F,H,W,C] (C = 3 or 4,
 * values in [0,1]); Ks[F,4] = (fx,fy,cx,cy) and c2ws[F,12] (row-major 3x4) are DEVICE arrays.  fid >= 0: all rays
 * from that frame (single-frame / vanilla mode); fid < 0: frame drawn per ray (mixed mode).  Pixels are uniform in
 * [w0,w1) x [h0,h1) (the precrop window, :119-127); RGBA is composited on white when white_bkgd (:129-132); rays
 * use pixel_center=True (:181-188).  Outputs: rgb[B,3], pixels_xy[B,2] [opt], fids_out[B] [opt] and the 6-tuple
 * of nsb_camera_rays.  Draws come from Philox(seed, step). */
int nsb_sample_pixel_batch(const float* images, int F, int H, int W, int C, const float* Ks, const float* c2ws, int fid,
                           int h0, int h1, int w0, int w1, int white_bkgd, int convention, int as_ndc, float near_plane,
                           int64_t B, uint64_t seed, uint64_t step, float* rgb, float* pixels_xy, int* fids_out,
                           float* o_world, float* d_world_unit, float* d_world_norm, float* o_march, float* d_march_unit,
                           float* d_march_norm, void* stream);

/* Eval output path (SURVEY section 8f rank 4): what ValidationRenderer does with a rendered frame,
 * utils/validation_renderer.py:485-533 with save_rgb_png / save_gray_png (utils/render_utils.py:28-47) and _compute_psnr
 * (:171-196), without leaving the device: rgb8[n,3] / acc8[n] / depth8[n] = (clamp(x,0,1) * 255 + 0.5) truncated to uint8,
 * depth first mapped to clamp((depth - fp32(near)) / fp32(far - near + 1e-8)) with a true division, bit for bit what torch computes
 * from Python-double near/far (or used as is when use_ndc); any output may be NULL.
 * With gt_rgb[n,3] (and optional mask[n], 1 = valid): psnr_out[0] = -10 log10(max(mse, 1e-10)), psnr_out[1] = mse with
 * mse = sum(mask * diff^2) / max(3 * sum(mask), 1e-8) over clamped values; psnr_scratch = 2 doubles of device scratch. */
int nsb_frame_output(const float* rgb, const float* acc, const float* depth, int64_t n, double depth_near, double depth_far,
                     int use_ndc, uint8_t* rgb8, uint8_t* acc8, uint8_t* depth8, const float* gt_rgb, const float* mask,
                     double* psnr_scratch, float* psnr_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NSB_H_ */
