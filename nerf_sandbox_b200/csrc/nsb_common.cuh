// Shared helpers for the libnsb kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/nsb.h"

namespace nsb {

// ---- launch bookkeeping -------------------------------------------------------------------------
extern int64_t g_launches;          // nsb_launch_count()
extern char g_cuda_err[256];
int check_launch(const char* what);  // cudaGetLastError -> NSB_E_CUDA
// Device-resident step counter of the call in progress (nsb_train_step only, else null): kernels that draw random numbers
// shift their Philox stream by 8 * (*g_step_dev), so a captured CUDA graph draws fresh numbers on every replay.
extern thread_local const uint64_t* g_step_dev;
extern thread_local uint64_t* g_pack_counter;
int num_sms();
int check_arch();                   // field_tc.cu: NSB_E_ARCH unless the current device is sm_100 (tcgen05 kernels)

#define NSB_LAUNCH_CHECK(name)                        \
    do {                                              \
        ++::nsb::g_launches;                          \
        int _e = ::nsb::check_launch(name);           \
        if (_e) return _e;                            \
    } while (0)

#define NSB_TRY(expr)          \
    do {                       \
        int _e = (expr);       \
        if (_e) return _e;     \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- Philox4x32-10 (counter based; one call -> 4 x 32 random bits) --------------------------------
__host__ __device__ inline void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                             uint32_t k0, uint32_t k1) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}
__host__ __device__ inline uint4 philox4(uint64_t seed, uint64_t stream_id, uint64_t idx) {
    uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32), c2 = (uint32_t)stream_id, c3 = (uint32_t)(stream_id >> 32);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// uniform in [0,1) on the 2^-24 grid (what torch.rand yields for fp32)
__host__ __device__ inline float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
__device__ inline float philox_uniform(uint64_t seed, uint64_t stream_id, uint64_t idx) {
    uint4 r = philox4(seed, stream_id, idx >> 2);
    uint32_t w = (idx & 3) == 0 ? r.x : (idx & 3) == 1 ? r.y : (idx & 3) == 2 ? r.z : r.w;
    return u01(w);
}
// one N(0,1) draw per index (Box-Muller on two words of the same Philox block)
__device__ inline float philox_normal(uint64_t seed, uint64_t stream_id, uint64_t idx) {
    uint4 r = philox4(seed, stream_id, idx >> 1);
    uint32_t a = (idx & 1) ? r.z : r.x, b = (idx & 1) ? r.w : r.y;
    float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0,1]
    float u2 = u01(b);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// N(0,1) for the sigma regulariser (render_utils.py:240): a 32-bit counter hash (two murmur3-style finalisers, one
// single-cycle IMAD each) + fast Box-Muller on MUFU (lg2 / sqrt / cos) -- ~22 instructions per draw where a Philox-10 block
// costs ~100; statistical quality is ample for additive training noise.  The compositor's forward and backward regenerate the
// same draw from (seed, stream, sample index).
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    return x;
}
// single-MUFU approximations (flush-to-zero variants need no denormal fix-up code around the MUFU)
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sqrt_approx(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float cos_approx(float x) { float y; asm("cos.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sin_approx(float x) { float y; asm("sin.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// the part of the hash key that does not depend on the low word of the index
__device__ __forceinline__ uint32_t hash_key(uint64_t seed, uint64_t stream_id, uint64_t idx) {
    return (uint32_t)seed ^ (uint32_t)(seed >> 32) * 0x9E3779B1u ^ (uint32_t)stream_id * 0x85EBCA77u ^
           (uint32_t)(stream_id >> 32) * 0xC2B2AE3Du ^ (uint32_t)(idx >> 32) * 0x27D4EB2Fu;
}
// Box-Muller on two independent hashes of the index: n0 = r cos(t), n1 = r sin(t), r = sqrt(-2 ln u1), t = 2 pi u2
__device__ __forceinline__ void hash_normal_pair(uint32_t key, uint32_t idx_lo, float& n0, float& n1) {
    const uint32_t a = mix32(idx_lo * 0x9E3779B1u + key);
    const uint32_t b = mix32(idx_lo * 0x7FEB352Du + (key ^ 0x68E31DA4u));
    const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0,1]
    const float t = (float)(b >> 8) * (6.2831853071795865f / 16777216.0f);
    const float r = sqrt_approx(-1.3862943611198906f * lg2_approx(u1));  // -2 ln u1 = -2 ln2 lg2(u1)
    n0 = r * cos_approx(t); n1 = r * sin_approx(t);
}
__device__ __forceinline__ float hash_normal(uint64_t seed, uint64_t stream_id, uint64_t idx) {
    float n0, n1;
    hash_normal_pair(hash_key(seed, stream_id, idx), (uint32_t)idx, n0, n1);
    return n0;
}

// ---- warp helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// ATen linspace(0,1,n)[i] in fp32 (symmetric fill; the upper half is one fused multiply-add)
__host__ __device__ inline float linspace01(int i, int n) {
    if (n <= 1) return 0.0f;
    const float step = 1.0f / (float)(n - 1);
    if (i < n / 2) return step * (float)i;
#ifdef __CUDA_ARCH__
    return __fmaf_rn(-step, (float)(n - 1 - i), 1.0f);
#else
    return (float)(1.0 - (double)step * (double)(n - 1 - i));
#endif
}

// ---- NeRF(63,27,8,256,4) geometry ---------------------------------------------------------------------
constexpr int kHidden = 256;
constexpr int kPosDim = 63, kPosPad = 64;
constexpr int kDirDim = 27;
constexpr int kSkipIn = 319, kSkipPad = 320;     // [h(256) | gamma(x)(63) | 0]
constexpr int kColorIn = 283, kColorPad = 288;   // [feat(256) | gamma(d)(27) | 0...]
constexpr int kColorHidden = 128;
constexpr int kNumGemmLayers = 10;               // mlp.0..7, feature, color_fc  (sigma_out/color_out are "heads")

struct LayerDesc { int N, K, Kpad; int64_t w_off, b_off; };   // offsets into the flat state_dict-ordered params
// index: 0..7 trunk, 8 feature, 9 sigma_out, 10 color_fc, 11 color_out
__host__ __device__ inline LayerDesc layer_desc(int l) {
    const int Ns[12] = {256, 256, 256, 256, 256, 256, 256, 256, 256, 1, 128, 3};
    const int Ks[12] = {63, 256, 256, 256, 319, 256, 256, 256, 256, 256, 283, 128};
    const int Kp[12] = {64, 256, 256, 256, 320, 256, 256, 256, 256, 256, 288, 128};
    int64_t off = 0;
    for (int i = 0; i < l; ++i) off += (int64_t)Ns[i] * Ks[i] + Ns[i];
    LayerDesc d; d.N = Ns[l]; d.K = Ks[l]; d.Kpad = Kp[l]; d.w_off = off; d.b_off = off + (int64_t)Ns[l] * Ks[l];
    return d;
}

// One layer GEMM of the fp32 mode, C[m,n] = sum_k A(m,k) * B(n,k), with the epilogue of its role (field_split.cu: on the
// tensor cores with bf16-split operands).
// AT = false: A stored [m][k] (k contiguous), AT = true: A stored [k][m]; same for BT and B.
enum { EPI_FWD = 0, EPI_DGRAD = 1, EPI_WGRAD = 2 };
struct GemmArgs {
    const float* A; int64_t lda;
    const float* B; int64_t ldb;
    float* C; int64_t ldc;
    int64_t Mdim, Ndim, Kdim;           // Kdim = contraction length
    const float* bias; int relu;        // FWD
    const float* mask; int64_t ldm;     // DGRAD: multiply by (mask > 0)
    const float* addend; int64_t ldadd; // DGRAD: += addend
    int n_valid;                        // WGRAD: columns < n_valid are written; DGRAD: when > 0, only columns < n_valid are
                                        //   written (and addend read), with scalar accesses: C / addend of any leading dimension
    int64_t k_per_split;                // WGRAD: contraction rows per split
    float* colsum;                      // WGRAD: += column sums of A (the bias gradient), or null
    const uint8_t* b_img;               // FWD / DGRAD: pre-split term images of B (split_pack), or null
};
// field_split.cu: role = EPI_* (FWD: A, B k-contiguous; DGRAD: B stored [k][n]; WGRAD: both stored [k][.], split-K with atomics)
int split_gemm(const GemmArgs& g, int role, cudaStream_t st);
size_t split_image_bytes(int n_rows, int k_len);                       // one weight matrix as a B operand: n_rows x k_len, 3 terms
int split_pack(const float* params, void* packed, cudaStream_t st);  // writes every split_fwd / split_dgrad image of a net

// Packed weights of one net (nsb_pack_weights): [fp32 padded section | bf16 tensor-core section]
struct PackedLayout {
    size_t f32_w[12], f32_b[12];   // byte offsets; rows padded to Kpad floats
    size_t bf16_off;               // start of the bf16 image (layout owned by field_tc.cu)
    size_t bf16_bytes;
    size_t split_fwd[12], split_dgrad[12];   // bf16 term images of the weights for the fp32 mode's tensor-core GEMMs (field_split.cu)
    size_t split_dinput[3];                   // ... and of the transposed input slices W_0[:, 0:63], W_4[:, 256:319], W_cfc[:, 256:283]
    size_t split_off, split_bytes;
    size_t total;
};
PackedLayout packed_layout();
size_t tc_packed_bytes();          // field_tc.cu

}  // namespace nsb
