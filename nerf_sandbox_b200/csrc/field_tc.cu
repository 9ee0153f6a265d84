// K1 (bf16 tensor-core mode) -- positional encoder + NeRF MLP as ONE persistent tcgen05 kernel per pass.
//
// Clusters of two CTAs (one per SM, cta_group::2) walk 128-point tiles, two tiles per CTA at a time.  Per tile, the chain
//     gamma(x) -> mlp.0..7 (skip concat at layer 4) -> feature -> color_fc -> heads
// runs without touching HBM for activations:
//   * A operand (activations, bf16) lives in shared memory in the tcgen05 canonical K-major layout (8x16 B core matrices,
//     no swizzle); the epilogue of layer l writes the A operand of layer l+1 in place;
//   * B operand (weights, bf16) is pre-packed by nsb_pack_weights in exactly that shared-memory image, ordered so that the
//     half of a K=32 slab one CTA of the pair needs (N/2 weight rows) is one contiguous 8 KB block; the TMA engine streams
//     it through an 8-stage ring with tensor-map loads whose complete_tx lands on the LEADER CTA's mbarrier;
//   * one tcgen05.mma spans both SMs: M = 256 = the tiles of the two CTAs, each CTA supplies half of B; accumulators (fp32)
//     live in each CTA's own TMEM: 2 tiles x 256 columns = all 512 columns;
//   * roles per CTA: warp 0 = TMA producer, warp 1 = MMA issuer (leader CTA only, one elected thread; commits are multicast
//     to both CTAs), warps 2-3 = per-tile helpers in training (proxy fence, hand-off, stash copy), warps 4-7 / 8-11 =
//     epilogue groups of tile A / tile B (thread == accumulator row: tcgen05.ld 32x32b, bias + ReLU, bf16 pack,
//     conflict-free st.shared).  While one tile's epilogue drains TMEM the tensor cores work on the other tile; a layer's
//     slabs are fetched once and used by tile A, then tile B;
//   * sigma_out (256->1) and color_out (128->3) are CUDA-core dot products inside the epilogues of layer 7 and color_fc
//     (fp32), so raw [r,g,b,sigma] leaves the chip as one float4 per point.
// Training adds a bf16 stash of every layer input (tile images + 1-bit ReLU masks) for the backward kernels: the dgrad chain
// (same CTA-pair machinery on transposed weight images) and wgrad (tile images as MN-major operands, accumulators resident in
// TMEM across all tiles of a CTA).  DESIGN.md section 4 has the measurements behind each of these choices.
#include <cuda.h>            // CUtensorMap (types only; the encoder is fetched with cudaGetDriverEntryPoint)
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdio>
#include <mutex>
#include "nsb_common.cuh"
#include "tc_ptx.cuh"

namespace nsb {
namespace tc {

constexpr int TILE_M = 128;
constexpr int kStageBytes = 16384;              // K=32 x N=256 bf16
constexpr int kStages = 4;
constexpr int kActBytes = TILE_M * 256 * 2;     // 65536
constexpr int kGxBytes = TILE_M * 64 * 2;       // 16384 (gamma(x), later gamma(d))
constexpr int kSmemAct = 0;
constexpr int kSmemGx = 2 * kActBytes;                      // 131072
constexpr int kSmemRing = kSmemGx + 2 * kGxBytes;           // 163840
constexpr int kSmemBar = kSmemRing + kStages * kStageBytes; // 229376
constexpr int kSmemBias = kSmemBar + 256;                   // 2 x 1 KB: per epilogue group, the current layer's bias
constexpr int kSmemBytes = kSmemBias + 2048;
constexpr int kThreads = 384;
// forward kernel, CTA pair: a ring stage holds this CTA's half of a K=32 slab (N/2 weight rows) -> twice the stages
constexpr int kStages2 = 8;
constexpr int kStageBytes2 = kStageBytes / 2;
static_assert(8 * (3 * kStages2 + 6) + 4 <= 256, "barrier block overflow");
constexpr int kNumMmaLayers = 10;               // mlp.0..7, feature, color_fc
constexpr uint32_t kTmemCols = 512;

// bf16 image offsets (bytes) of the 10 MMA layers: [K/8][N][8] bf16 each
__constant__ uint32_t c_layer_ofs[kNumMmaLayers] = {0,      32768,  163840, 294912, 425984,
                                                    589824, 720896, 851968, 983040, 1114112};
constexpr uint32_t kWeightImageBytes = 1114112 + 288 * 128 * 2;   // 1,187,840
// fp32 tail: biases of the 10 MMA layers (9x256 + 128), w_sigma[256], b_sigma, Wo[3][128], bo[3]
constexpr uint32_t kBiasOfs = kWeightImageBytes;                  // floats from here
constexpr int kBiasFloats = 9 * 256 + 128;
constexpr int kWsigOfs = kBiasFloats;                             // float index within the tail
constexpr int kBsigOfs = kWsigOfs + 256;
constexpr int kWoOfs = kBsigOfs + 4;                              // keep 16B alignment
constexpr int kBoOfs = kWoOfs + 384;
constexpr int kTailFloats = kBoOfs + 4;
// transposed images for the dgrad chain (contraction over OUT features, first 256 IN features as N):
//   m=0 color_fc^T (K=128) | m=1 feature^T | m=2..8 mlp.7^T .. mlp.1^T (K=256 each); element (j, n) at [n/8][j][8]
constexpr uint32_t kTImgOfs = ((kBiasOfs + kTailFloats * 4 + 255) / 256) * 256;
constexpr int kNumDgradLayers = 9;
__host__ __device__ inline uint32_t dgrad_layer_ofs(int m) { return kTImgOfs + (m == 0 ? 0u : 65536u + (uint32_t)(m - 1) * 131072u); }
// fp16 copy of the forward images (same layout as the bf16 ones at offset 0) for the inference kernel
constexpr uint32_t kF16ImgOfs = kTImgOfs + 65536 + 8 * 131072;
static_assert(kF16ImgOfs % 256 == 0 && kWeightImageBytes % 256 == 0, "images are addressed as rows of 256 B");
// low halves of the fp16 SPLIT  w = hi + lo  (hi = the fp16 image above, lo = fp16(w - hi)) for the fp32-accurate forward
constexpr uint32_t kF16LoImgOfs = kF16ImgOfs + kWeightImageBytes;
// B operands of the input-gradient products (field_dinput_kernel), bf16 K-major images [k/8][rows][8] with k = out feature:
//   W_0[:, 0:63]^T (64 rows, K = 256) | W_4[:, 256:319]^T (64 rows, K = 256) | W_cfc[:, 256:283]^T (32 rows, K = 128); padding zero
constexpr uint32_t kDinImgOfs = kF16LoImgOfs + kWeightImageBytes;
constexpr uint32_t kDinPos0 = 0, kDinPos4 = 32768, kDinDir = 65536, kDinImgBytes = 73728;
constexpr uint32_t kPackedTcBytes = kDinImgOfs + kDinImgBytes;

__host__ __device__ inline int layer_nslabs(int l) { return l == 0 ? 2 : (l == 4 ? 10 : (l == 9 ? 9 : 8)); }
__host__ __device__ inline int layer_N(int l) { return l == 9 ? 128 : 256; }
__host__ __device__ inline int layer_bias_ofs(int l) { return l * 256; }

// Number formats (instruction-descriptor bits [7,10) = A, [10,13) = B: 0 = f16, 1 = bf16; accumulation is fp32 throughout).
//  * INFERENCE forward (no stash: eval frames, no-grad passes): fp16 operands -- weights, gamma(x), gamma(d), activations.
//    11 significant bits, what the reference computes in under its CUDA autocast (utils/render_utils.py:334-335), 8x finer
//    than bf16; the positional encoding's high-frequency features and the 9-layer chain are where that shows in a render.
//  * TRAINING forward + backward: bf16 everywhere.  The stash is the forward's own operand images and wgrad multiplies them
//    with dY tiles, which need fp32's exponent range (no loss scaling here); kind::f16 MMAs with DIFFERENT A and B formats
//    trap with "illegal instruction" on B200 (measured: dgrad with A = bf16, B = fp16), so both operands of every backward
//    MMA -- hence the stashed activations, hence the training forward -- are bf16.
constexpr uint32_t kFmtF16 = 0u, kFmtBF16 = 1u;
// kind::f16 instruction descriptor of a CTA pair: D = f32, both operands K-major, M = 256 (128 rows per CTA)
__device__ __forceinline__ uint32_t make_idesc2(int N, uint32_t a_fmt, uint32_t b_fmt) {
    return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)((2 * TILE_M) >> 4) << 24);
}

// {lo = relu(a), hi = relu(b)} as bf16x2 in one instruction
__device__ __forceinline__ uint32_t pack_bf16_relu(float a, float b) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&t);
}
// fp16 pair {lo = a, hi = b}, saturating at +-65504 instead of overflowing to inf; _relu clamps negatives to +0 first
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ uint32_t pack_f16_relu(float a, float b) {
    uint32_t d;
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
template <bool F16> __device__ __forceinline__ uint32_t pack2(float a, float b) { return F16 ? pack_f16(a, b) : pack_bf16(a, b); }
template <bool F16> __device__ __forceinline__ uint32_t pack2_relu(float a, float b) { return F16 ? pack_f16_relu(a, b) : pack_bf16_relu(a, b); }

// 16 ReLU'd bf16 outputs held as 8 packed words -> 16 mask bits: bit j (even column 2j) and bit 16+j (odd column 2j+1).
// __vsetne2 gives 0x0001 per non-zero half-word; one multiply-add per word shifts it into place.
__device__ __forceinline__ uint32_t relu_bits16(const uint32_t (&w)[8]) {
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += __vsetne2(w[j], 0u) << j;
    return s;
}
// the 0xFFFF-per-half AND mask of packed word j of a 16-column chunk, from its bit field (already shifted to bit 0)
__device__ __forceinline__ uint32_t relu_mask_word(uint32_t bits16, int j) { return ((bits16 >> j) & 0x00010001u) * 0xFFFFu; }

// ---- epilogue column loop, specialised per layer kind (branch-free inner loop) ---------------------------
// KIND 0: bias + ReLU -> bf16 A operand (mlp.0..6)          KIND 1: same + sigma_out head on the fp32 values (mlp.7)
// KIND 2: bias only (feature)                              KIND 3: bias + ReLU + color_out head (color_fc, N=128);
//                                                                  writes c to smem only when WRITE (training stash)
__device__ __forceinline__ void st_chunk(uint32_t base, int k8, int r, uint32_t a, uint32_t b, uint32_t c, uint32_t d);
__device__ __forceinline__ void st_chunk_g(uint8_t* grow, int k8, uint32_t a, uint32_t b, uint32_t c, uint32_t d);
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
template <int KIND, bool MASK>
__device__ __forceinline__ void epi_chunk16(const uint32_t (&v)[16], int c0, const float4 (&bias)[4], uint32_t act, int r, float& sig,
                                            float (&rgb)[3], float hw0, float hw1, float hw2, uint32_t& mbits) {
    float f[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        f[4 * j] = __uint_as_float(v[4 * j]) + bias[j].x; f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + bias[j].y;
        f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + bias[j].z; f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + bias[j].w;
    }
    if (KIND == 1 || KIND == 3) {
        const int src0 = c0 & 16;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            f[j] = fmaxf(f[j], 0.f);
            if (KIND == 1) sig = fmaf(f[j], __shfl_sync(0xffffffffu, hw0, src0 + j), sig);
            if (KIND == 3) {
                rgb[0] = fmaf(f[j], __shfl_sync(0xffffffffu, hw0, src0 + j), rgb[0]);
                rgb[1] = fmaf(f[j], __shfl_sync(0xffffffffu, hw1, src0 + j), rgb[1]);
                rgb[2] = fmaf(f[j], __shfl_sync(0xffffffffu, hw2, src0 + j), rgb[2]);
            }
        }
    }
    if (KIND != 3 || MASK) {          // color_fc output goes to shared memory only for the training stash
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = KIND == 0 ? pack2_relu<!MASK>(f[2 * j], f[2 * j + 1]) : pack2<!MASK>(f[2 * j], f[2 * j + 1]);
        st_chunk(act, (c0 >> 3), r, w[0], w[1], w[2], w[3]);
        st_chunk(act, (c0 >> 3) + 1, r, w[4], w[5], w[6], w[7]);
        if (KIND != 2 && MASK) mbits = relu_bits16(w);            // training: ReLU mask bits of these 16 outputs
    }
}
// MASK = training: mask words kept in registers and written once after the loop to gmask (this row's 32 B of the layer's
// mask slot; null for rows of a tile past the end)
template <int KIND, bool MASK>
__device__ __forceinline__ void epi_columns(uint32_t tmem_row, uint32_t sbias, uint32_t act, int r, int lane, const float* __restrict__ tail,
                                            float& sig, float (&rgb)[3], uint32_t* gmask) {
    constexpr int N = KIND == 3 ? 128 : 256;
    float hw0 = 0.f, hw1 = 0.f, hw2 = 0.f;          // lane-held 32-wide slice of the head weights
    if (KIND == 1) hw0 = __ldg(tail + kWsigOfs + lane);
    if (KIND == 3) { hw0 = __ldg(tail + kWoOfs + lane); hw1 = __ldg(tail + kWoOfs + 128 + lane); hw2 = __ldg(tail + kWoOfs + 256 + lane); }
    uint32_t mw[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    uint32_t va[16], vb[16];
    tc_ld16(tmem_row, va);
#pragma unroll 1
    for (int c0 = 0; c0 < N; c0 += 32) {
        // bias of these 32 columns: issued BEFORE the TMEM wait so the shared-memory latency hides behind it
        float4 ba[4], bb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { ba[j] = lds_f4(sbias + 4u * (uint32_t)(c0 + 4 * j)); bb[j] = lds_f4(sbias + 4u * (uint32_t)(c0 + 16 + 4 * j)); }
        float n0 = 0.f, n1 = 0.f, n2 = 0.f;
        if (KIND == 1 && c0 + 32 < N) n0 = __ldg(tail + kWsigOfs + c0 + 32 + lane);
        if (KIND == 3 && c0 + 32 < N) {
            n0 = __ldg(tail + kWoOfs + c0 + 32 + lane); n1 = __ldg(tail + kWoOfs + 128 + c0 + 32 + lane);
            n2 = __ldg(tail + kWoOfs + 256 + c0 + 32 + lane);
        }
        // consumers pinned BEHIND the next TMEM load: the pin follows the tcgen05.ld in program order, so this chunk's
        // math cannot be hoisted above the issue of the next load
        tc_wait_ld();
        tc_ld16(tmem_row + (uint32_t)c0 + 16u, vb);
        pin16(va);
        uint32_t m0 = 0, m1 = 0;
        epi_chunk16<KIND, MASK>(va, c0, ba, act, r, sig, rgb, hw0, hw1, hw2, m0);
        tc_wait_ld();
        tc_ld16(tmem_row + (uint32_t)(c0 + 32 < N ? c0 + 32 : c0), va);      // last iteration: harmless re-read
        pin16(vb);
        epi_chunk16<KIND, MASK>(vb, c0 + 16, bb, act, r, sig, rgb, hw0, hw1, hw2, m1);
        if (MASK) {                                       // one mask word per 32 columns, kept in registers until the end
            const uint32_t m = m0 | (m1 << 8);
#pragma unroll
            for (int k = 0; k < 8; ++k) mw[k] = (c0 >> 5) == k ? m : mw[k];
        }
        hw0 = n0; hw1 = n1; hw2 = n2;
    }
    if (MASK && gmask) {
        reinterpret_cast<uint4*>(gmask)[0] = make_uint4(mw[0], mw[1], mw[2], mw[3]);
        reinterpret_cast<uint4*>(gmask)[1] = make_uint4(mw[4], mw[5], mw[6], mw[7]);
    }
}

// ---- kernel parameters --------------------------------------------------------------------------------
struct FwdParams {
    const float* rays_o; const float* rays_d; const float* z; const float* ray_norm; const float* viewdirs;   // FROM_ENC=false
    const float* enc_pos; const float* enc_dir;                                                                  // FROM_ENC=true
    const uint8_t* packed;        // bf16 image + fp32 tail
    float* raw;                   // [Q,4]
    uint8_t* stash;               // training: per tile, images of the layer inputs (see StashLayout); else null
    float* dbg; int dbg_layer;    // debug: post-activation fp32 of one layer, [Q,256]
    unsigned long long* cyc;      // debug: per-role wait/busy cycle counters of CTA 0 (16 x u64), or null
    int64_t Q; int N;             // points, samples per ray
    int64_t num_tiles;
    // the packed buffer as rows of 256 B: boxes of 32 rows (8 KB half slab, N = 256) and 16 rows (4 KB, N = 128)
    alignas(64) CUtensorMap tm8;
    alignas(64) CUtensorMap tm4;
};

// Stash of one tile (bytes), every block a shared-memory image ([K/8][128 rows][8] bf16):
//   gx (K=64) 16384 | h1..h8 (inputs of mlp.1..7 and of feature/sigma; K=256) 8 x 65536 | feat (K=256) 65536 |
//   gd (K=32) 8192 | c (color_fc output, K=128) 32768
constexpr size_t kStashGx = 0, kStashH = 16384, kStashFeat = kStashH + 8 * 65536, kStashGd = kStashFeat + 65536,
                 kStashC = kStashGd + 8192,
                 // ReLU masks, one bit per element: slot s (0..7 = h1..h8, 8 = c), row r, 8 words (32 B per row and slot).
                 // Word w covers columns [32w, 32w+32): bit (8*(c/16%2) + (c%16)/2) + 16*(c%2)  -- see relu_bits16().
                 kStashMask = kStashC + 32768, kStashTile = kStashMask + 9 * 128 * 32;   // 684,032 B / tile = 5344 B / point
// Gradient stash of one tile, written by the dgrad chain and read by wgrad (same image layout):
//   dY_9 (d pre-activation of color_fc, K=128) 32768 | dY_8 (d feature out) | dY_7 .. dY_0 (d pre-act of mlp.7..0), 65536 each
constexpr size_t kDstashTile = 32768 + 9 * 65536;                           // 622,592 B / tile = 4864 B / point
__host__ __device__ inline size_t dstash_ofs(int k) { return k == 9 ? 0 : 32768 + (size_t)(8 - k) * 65536; }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// ---- operand hand-off (epilogue group -> MMA issuer) and stash write-out --------------------------------
// Two things must not be done by the 128 epilogue threads themselves:
//  * the generic->async proxy fence that tcgen05.mma needs before it reads an A operand written with st.shared
//    (ptxas emits MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC for it, and the MEMBAR waits for every memory operation the thread
//    has in flight), and
//  * the stash stores to global memory: any st.global inside the TMEM column loop -- even one 4-byte store per 32
//    columns -- stretched the loop from ~2.9k to ~5.2k cycles per layer (measured with the per-role cycle counters),
//    which made the training forward 1.6x slower than the same kernel without a stash.
// So the epilogue threads only write shared memory and bar.arrive on a named barrier; a helper warp per tile (warps 2, 3:
// no stores of their own) waits on that barrier, issues the proxy fence, arrives on the MMA issuer's mbarrier and lets the
// TMA engine copy the finished tile image to the stash (cp.async.bulk shared -> global).  Once the engine has read the
// tile the helper releases the group's "tile may be overwritten" barrier (named barrier 1+t, 128 + 32 threads).
constexpr int kHandoffBar = 3;          // named barriers 3 (tile A) and 4 (tile B): 128 arrivals + the helper warp
__device__ __forceinline__ void handoff_signal(int t) {
    tc_fence_before();
    named_bar_arrive(kHandoffBar + t, 160);
}
// helper side of one event: returns after the fence; lane 0 then arrives / stores
__device__ __forceinline__ void handoff_wait(int t) {
    named_bar_sync(kHandoffBar + t, 160);
    tc_fence_after();
    fence_async_smem();
    tc_fence_before();
}
// "this CTA's A tile t is in place": the leader's own tiles count on bar_in, the peer's on the leader's bar_pin
__device__ __forceinline__ void arrive_in(uint32_t crank, uint32_t bar_in, uint32_t bar_pin, int t) {
    if (crank == 0) mbar_arrive(bar_in + 8 * t); else mbar_arrive_remote(bar_pin + 8 * t, 0);
}
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// write 8 consecutive K elements (one 16-byte core-matrix row) of row r at K-chunk `k8`
__device__ __forceinline__ void st_chunk(uint32_t base, int k8, int r, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + (uint32_t)k8 * 2048u + (uint32_t)r * 16u), "r"(a), "r"(b),
                 "r"(c), "r"(d)
                 : "memory");
}

// the same 16-byte row chunk straight to the (d)stash image in global memory: per warp 32 rows x 16 B = 512 contiguous
// bytes per chunk -> fully coalesced 128-bit stores, no smem read-back, no barrier
__device__ __forceinline__ void st_chunk_g(uint8_t* grow, int k8, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    if (grow) *reinterpret_cast<uint4*>(grow + (size_t)k8 * 2048) = make_uint4(a, b, c, d);
}

// gamma(x) of this thread's point -> gx buffer (K=64: [x(3) | sin(2^k x_d) k-major (30) | cos (30) | 0])
template <bool F16>
__device__ __forceinline__ void encode_pos(uint32_t gx, int r, float px, float py, float pz, uint8_t* grow) {
    float e[64];
    e[0] = px; e[1] = py; e[2] = pz; e[63] = 0.f;
    float s[3], c[3];
    sincosf(px, &s[0], &c[0]); sincosf(py, &s[1], &c[1]); sincosf(pz, &s[2], &c[2]);
#pragma unroll
    for (int k = 0; k < 10; ++k) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            e[3 + 3 * k + d] = s[d]; e[33 + 3 * k + d] = c[d];
            const float s2 = 2.0f * s[d] * c[d], c2 = fmaf(-2.0f * s[d], s[d], 1.0f);   // angle doubling
            s[d] = s2; c[d] = c2;
        }
    }
#pragma unroll
    for (int k8 = 0; k8 < 8; ++k8) {
        const uint32_t w0 = pack2<F16>(e[8 * k8], e[8 * k8 + 1]), w1 = pack2<F16>(e[8 * k8 + 2], e[8 * k8 + 3]),
                       w2 = pack2<F16>(e[8 * k8 + 4], e[8 * k8 + 5]), w3 = pack2<F16>(e[8 * k8 + 6], e[8 * k8 + 7]);
        st_chunk(gx, k8, r, w0, w1, w2, w3);
        st_chunk_g(grow, k8, w0, w1, w2, w3);
    }
}
// gamma(d) -> first 4 K-chunks of the gx buffer (K=32: [v(3) | sin (12) | cos (12) | 0 x5])
template <bool F16>
__device__ __forceinline__ void encode_dir(uint32_t gx, int r, float vx, float vy, float vz, uint8_t* grow) {
    float e[32];
#pragma unroll
    for (int i = 27; i < 32; ++i) e[i] = 0.f;
    e[0] = vx; e[1] = vy; e[2] = vz;
    float s[3], c[3];
    sincosf(vx, &s[0], &c[0]); sincosf(vy, &s[1], &c[1]); sincosf(vz, &s[2], &c[2]);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            e[3 + 3 * k + d] = s[d]; e[15 + 3 * k + d] = c[d];
            const float s2 = 2.0f * s[d] * c[d], c2 = fmaf(-2.0f * s[d], s[d], 1.0f);
            s[d] = s2; c[d] = c2;
        }
    }
#pragma unroll
    for (int k8 = 0; k8 < 4; ++k8) {
        const uint32_t w0 = pack2<F16>(e[8 * k8], e[8 * k8 + 1]), w1 = pack2<F16>(e[8 * k8 + 2], e[8 * k8 + 3]),
                       w2 = pack2<F16>(e[8 * k8 + 4], e[8 * k8 + 5]), w3 = pack2<F16>(e[8 * k8 + 6], e[8 * k8 + 7]);
        st_chunk(gx, k8, r, w0, w1, w2, w3);
        st_chunk_g(grow, k8, w0, w1, w2, w3);
    }
}
// materialised encodings (NeRF.forward boundary): copy a row of `n` floats, zero-padded to 8*chunks
template <bool F16>
__device__ __forceinline__ void copy_enc_row(uint32_t gx, int r, const float* __restrict__ src, int n, int chunks, uint8_t* grow) {
    for (int k8 = 0; k8 < chunks; ++k8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (8 * k8 + j < n && src) ? src[8 * k8 + j] : 0.f;
        const uint32_t w0 = pack2<F16>(v[0], v[1]), w1 = pack2<F16>(v[2], v[3]), w2 = pack2<F16>(v[4], v[5]), w3 = pack2<F16>(v[6], v[7]);
        st_chunk(gx, k8, r, w0, w1, w2, w3);
        st_chunk_g(grow, k8, w0, w1, w2, w3);
    }
}

// STASH = training: the kernel also writes the stash (p.stash) that the backward kernels read
template <bool FROM_ENC, bool STASH>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) field_fwd_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();           // 0 = leader (issues the pair's MMAs)
    // barriers: full[8] empty[8] in_ready[2] acc_full[2] peer_full[8] peer_in[2]; then the TMEM base address.
    // full/in_ready are local; empty/acc_full get the leader's multicast commits; peer_* (used in the leader only) are
    // arrived on by the peer's relay thread once the peer's half slab / A tile is in place.
    const uint32_t bar_full = sbase + kSmemBar, bar_empty = bar_full + 8 * kStages2, bar_in = bar_empty + 8 * kStages2,
                   bar_acc = bar_in + 16, bar_pfull = bar_acc + 16, bar_pin = bar_pfull + 8 * kStages2;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kSmemBar + 8 * (3 * kStages2 + 6));

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages2; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); mbar_init(bar_pfull + 8 * s, 1); }
        // inference (no stash): the 128 epilogue threads fence and arrive themselves; training: the tile's helper warp does
        for (int t = 0; t < 2; ++t) { mbar_init(bar_in + 8 * t, STASH ? 1 : 128); mbar_init(bar_acc + 8 * t, 1); mbar_init(bar_pin + 8 * t, STASH ? 1 : 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {   // TMEM allocation (whole SM: 2 tiles x 256 fp32 columns), collectively with the peer CTA's warp 2
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();          // the peer's barriers and TMEM exist before anything is sent its way
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int64_t num_pairs = (p.num_tiles + 1) / 2;
    // both CTAs of a cluster walk the weight stream in lockstep: same trip count (the leader's); a CTA whose pair index
    // falls off the end computes on stale tiles and stores nothing
    const int64_t first_pair = (int64_t)blockIdx.x - crank;
    const int64_t n_iter = first_pair < num_pairs ? (num_pairs - first_pair + gridDim.x - 1) / gridDim.x : 0;
    const float* tail = reinterpret_cast<const float*>(p.packed + kBiasOfs);

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        // (whole warp runs the uniform control flow; one lane issues -- keeps operands in uniform registers)
        {
            uint32_t stage = 0, round = 0;
            long long w_empty = 0; const long long t_begin = clock64();
            for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
                for (int l = 0; l < kNumMmaLayers; ++l) {
                    const uint32_t bytes = 32u * (uint32_t)layer_N(l) * 2u;
                    const int ns = layer_nslabs(l);
                    // a layer whose slabs fit the ring is fetched once and used by tile A, then by tile B; the two longer
                    // layers (the skip layer and color_fc) are streamed once per tile
                    for (int s2 = 0; s2 < (ns <= kStages2 ? ns : 2 * ns); ++s2) {
                        const int s = s2 >= ns ? s2 - ns : s2;
                        mbar_wait_t(bar_empty + 8 * stage, (round & 1) ^ 1, w_empty);
                        if (elect_one()) {
                            // this CTA's half of the slab: weight rows [crank * N/2, +N/2), contiguous in the packed image.
                            // Both halves complete on the leader's barrier, which therefore expects the whole slab.
                            const uint32_t half = bytes >> 1;
                            if (crank == 0) mbar_expect_tx(bar_full + 8 * stage, bytes);
                            tma_load_rows_to_leader(sbase + kSmemRing + stage * kStageBytes2, half == 8192u ? &p.tm8 : &p.tm4,
                                                    ((STASH ? 0u : kF16ImgOfs) + c_layer_ofs[l] + (uint32_t)s * bytes + crank * half) >> 8, bar_full + 8 * stage);
                        }
                        __syncwarp();
                        if (++stage == kStages2) { stage = 0; ++round; }
                    }
                }
            }
            if (p.cyc && blockIdx.x == 0 && lane == 0) { p.cyc[0] = (unsigned long long)w_empty; p.cyc[1] = (unsigned long long)(clock64() - t_begin); }
            if (p.cyc && blockIdx.x == 1 && lane == 0) { p.cyc[16] = (unsigned long long)w_empty; p.cyc[17] = (unsigned long long)(clock64() - t_begin); }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer ========================================
        // ONE elected thread runs the whole issue loop (elect.sync tells ptxas a single lane is live, so tcgen05 operands go
        // to uniform registers without per-lane waterfalls and there is no per-slab warp re-convergence).
        // Schedule: tile A's whole layer, then tile B's -- while one tile's epilogue drains TMEM the tensor core works on
        // the other tile; the layer's weight slabs are streamed once per tile.
        if (crank == 0 && elect_one()) {
            uint32_t stage = 0, round = 0, use = 0;   // use = layers completed (parity of in_ready / acc_full)
            long long w_in = 0, w_full = 0, w_pfull = 0, w_pin = 0; const long long t_begin = clock64();
            const uint64_t ahi = desc_hi(2048, 128);
            const uint32_t ring_lo = (sbase + kSmemRing) >> 4;
            // issue `n` K=32 slabs whose A operand starts at a_lo (descriptor address units of 16 B) into accumulator d_tmem.
            // wait: the slabs have not been seen yet (first use);  release: hand the stages back to the producers after use
            auto issue = [&](uint32_t a_lo, int n, bool first_overwrites, uint32_t d_tmem, uint64_t bhi, uint32_t b_step, uint32_t idesc,
                             uint32_t acc_bar, bool wait, bool release) {
                for (int s = 0; s < n; ++s, a_lo += 512u) {
                    if (wait) {
                        if (p.cyc) mbar_wait_t(bar_full + 8 * stage, round & 1, w_full); else mbar_wait(bar_full + 8 * stage, round & 1);
                        tc_fence_after();
                    }
                    const uint32_t b_lo = ring_lo + stage * (kStageBytes2 >> 4);
                    tc_mma2(d_tmem, ahi | (uint64_t)a_lo, bhi | (uint64_t)b_lo, idesc, (first_overwrites && s == 0) ? 0u : 1u);
                    tc_mma2(d_tmem, ahi | (uint64_t)(a_lo + 256u), bhi | (uint64_t)(b_lo + b_step), idesc, 1u);
                    if (acc_bar && s == n - 1) tc_commit2(acc_bar);
                    if (release) tc_commit2(bar_empty + 8 * stage);
                    if (++stage == kStages2) { stage = 0; ++round; }
                }
            };
            for (int64_t it = 0; it < n_iter; ++it) {
                for (int l = 0; l < kNumMmaLayers; ++l, ++use) {
                    const int N = layer_N(l);
                    const uint32_t idesc = make_idesc2(N, STASH ? kFmtBF16 : kFmtF16, STASH ? kFmtBF16 : kFmtF16);
                    const uint32_t lbo_b = (uint32_t)N * 8u;            // K-chunk stride inside a stage: N/2 rows x 16 B
                    const uint64_t bhi = desc_hi(lbo_b, 128);
                    const uint32_t b_step = (2u * lbo_b) >> 4;
                    // A-operand segments of the layer: n_act slabs from the activation buffer, then n_gx from the gamma buffer
                    const int n_act = l == 0 ? 0 : 8;
                    const int n_gx = l == 0 ? 2 : (l == 4 ? 2 : (l == 9 ? 1 : 0));
                    const bool shared = n_act + n_gx <= kStages2;       // slabs fetched once, used by tile A then tile B
                    const uint32_t stage0 = stage, round0 = round;
                    for (int t = 0; t < 2; ++t) {
                        if (p.cyc) mbar_wait_t(bar_in + 8 * t, use & 1, w_in); else mbar_wait(bar_in + 8 * t, use & 1);
                        { const long long t0 = clock64(); mbar_wait_cl(bar_pin + 8 * t, use & 1); w_pin += clock64() - t0; }
                        tc_fence_after();
                        if (shared && t == 1) { stage = stage0; round = round0; }
                        const bool wait = !shared || t == 0, release = !shared || t == 1;
                        const uint32_t d_tmem = tmem_base + (uint32_t)t * 256u;
                        const uint32_t act_lo = (sbase + kSmemAct + t * kActBytes) >> 4, gx_lo = (sbase + kSmemGx + t * kGxBytes) >> 4;
                        const uint32_t acc_bar = bar_acc + 8 * t;
                        if (n_act) issue(act_lo, n_act, true, d_tmem, bhi, b_step, idesc, n_gx ? 0u : acc_bar, wait, release);
                        if (n_gx) issue(gx_lo, n_gx, n_act == 0, d_tmem, bhi, b_step, idesc, acc_bar, wait, release);
                    }
                }
            }
            if (p.cyc && blockIdx.x == 0) {
                p.cyc[2] = (unsigned long long)w_in; p.cyc[3] = (unsigned long long)w_full; p.cyc[4] = (unsigned long long)(clock64() - t_begin);
                p.cyc[13] = (unsigned long long)w_pfull; p.cyc[14] = (unsigned long long)w_pin;
            }
        }
    } else if (STASH && (warp == 2 || warp == 3)) {
        // ============================ operand hand-off + stash write-out, one warp per tile ======================
        // events per pair: e0 = layer-0 input encoded; e1..e9 = output of layer e-1 in the activation tile (next A operand;
        // training: image of h_{e} / feat -> stash); training only: e10 = c (color_fc output) -> stash, feeds no MMA
        const int t = warp - 2;
        const uint32_t act = sbase + kSmemAct + t * kActBytes;
        const int n_events = kNumMmaLayers + 1;
        for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
            const int64_t tile = pair * 2 + t;
            uint8_t* stash_tile = tile < p.num_tiles ? p.stash + (size_t)tile * kStashTile : nullptr;
            for (int e = 0; e < n_events; ++e) {
                handoff_wait(t);
                if (lane == 0) {
                    if (e < kNumMmaLayers) arrive_in(crank, bar_in, bar_pin, t);
                    if (stash_tile && e >= 1) {
                        const int l = e - 1;
                        const size_t ofs = l <= 7 ? kStashH + (size_t)l * 65536 : (l == 8 ? kStashFeat : kStashC);
                        bulk_s2g(stash_tile + ofs, act, l == 9 ? 32768u : 65536u);
                        bulk_commit();
                        bulk_wait_read0();          // the engine has read the tile: it may be overwritten
                    }
                }
                __syncwarp();
                if (e < kNumMmaLayers) named_bar_arrive(1 + t, 160);      // release for the epilogue of layer e
            }
        }
        if (lane == 0) bulk_wait_all0();
    } else if (warp >= 4) {
        // ===================================== epilogue groups ===================================
        const int t = (warp - 4) >> 2;                 // tile of the pair: 0 = A, 1 = B
        const int r = (int)threadIdx.x - 128 - t * 128; // accumulator row == TMEM lane == point within the tile
        const uint32_t act = sbase + kSmemAct + t * kActBytes, gx = sbase + kSmemGx + t * kGxBytes;
        const uint32_t tmem_row = tmem_base + (uint32_t)t * 256u + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t use = 0;
        long long w_acc = 0, w_bar = 0, t_cols = 0; const long long t_begin = clock64();
        for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
            const int64_t tile = pair * 2 + t;
            const int64_t q = tile * TILE_M + r;
            const bool valid = tile < p.num_tiles && q < p.Q;
            const int64_t qc = valid ? q : 0;
            // training stash: gamma(x), gamma(d) and the mask words are stored from here; the activation tiles by the helper warp
            constexpr bool do_stash = STASH;
            uint8_t* stash_tile = do_stash && tile < p.num_tiles ? p.stash + (size_t)tile * kStashTile : nullptr;
            // row pointer into a stash block (or null): every 16-byte chunk written to smem is mirrored there
            auto srow = [&](size_t ofs) -> uint8_t* { return stash_tile ? stash_tile + ofs + (size_t)r * 16 : nullptr; };
            // ---- layer-0 input: gamma(x) ----
            float vdir[3] = {0.f, 0.f, 1.f};
            if (FROM_ENC) {
                copy_enc_row<!STASH>(gx, r, valid ? p.enc_pos + qc * kPosDim : nullptr, kPosDim, 8, srow(kStashGx));
            } else {
                const int64_t b = qc / p.N;
                const float zz = valid ? p.z[qc] : 0.f;
                const float zm = p.ray_norm ? zz * p.ray_norm[b] : zz;
                const float px = fmaf(p.rays_d[b * 3 + 0], zm, p.rays_o[b * 3 + 0]);
                const float py = fmaf(p.rays_d[b * 3 + 1], zm, p.rays_o[b * 3 + 1]);
                const float pz = fmaf(p.rays_d[b * 3 + 2], zm, p.rays_o[b * 3 + 2]);
                encode_pos<!STASH>(gx, r, px, py, pz, srow(kStashGx));
                const float* vs = p.viewdirs ? p.viewdirs : p.rays_d;
                const float vx = vs[b * 3 + 0], vy = vs[b * 3 + 1], vz = vs[b * 3 + 2];
                const float inv = 1.0f / fmaxf(sqrtf(vx * vx + vy * vy + vz * vz), 1e-12f);
                vdir[0] = vx * inv; vdir[1] = vy * inv; vdir[2] = vz * inv;
            }
            if (do_stash) handoff_signal(t); else { fence_async_smem(); arrive_in(crank, bar_in, bar_pin, t); }
            float sig = 0.f, rgb[3] = {0.f, 0.f, 0.f};
            const uint32_t sbias = sbase + kSmemBias + (uint32_t)t * 1024u;      // this group's bias staging (256 fp32)
            const bool want_dbg = p.dbg != nullptr;
            for (int l = 0; l < kNumMmaLayers; ++l, ++use) {
                const int N = layer_N(l);
                // While the MMAs of this layer run: fetch its bias (coalesced, one or two floats per thread) and the first
                // lane-held slice of the head weights.  Nothing inside the column loop touches global memory.
                const float b_lo = __ldg(tail + layer_bias_ofs(l) + r);
                const float b_hi = N == 256 ? __ldg(tail + layer_bias_ofs(l) + 128 + r) : 0.f;
                float hw0 = 0.f, hw1 = 0.f, hw2 = 0.f;      // l==7: w_sigma[32g+lane];  l==9: Wo[ch][32g+lane]
                if (l == 7) hw0 = __ldg(tail + kWsigOfs + lane);
                if (l == 9) { hw0 = __ldg(tail + kWoOfs + lane); hw1 = __ldg(tail + kWoOfs + 128 + lane); hw2 = __ldg(tail + kWoOfs + 256 + lane); }
                mbar_wait_t(bar_acc + 8 * t, use & 1, w_acc);
                tc_fence_after();
                // group barrier 1: everyone is past the previous layer's reads of sbias, and the helper warp has released the
                // activation tile (its previous image has been read by the stash copy)
                const long long tb0 = clock64();
                named_bar_sync(1 + t, do_stash ? 160 : 128);
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(sbias + 4u * (uint32_t)r), "f"(b_lo) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(sbias + 512u + 4u * (uint32_t)r), "f"(b_hi) : "memory");
                named_bar_sync(1 + t, 128);                 // group barrier 2: bias visible
                const long long tc0 = clock64();
                w_bar += tc0 - tb0;
                const bool relu = l != 8;
                const bool need_f32 = l == 7 || l == 9 || (want_dbg && l == p.dbg_layer);
                const bool write_act = l != 9;              // next layer's A operand, in place
                // column loop, 16 accumulator columns at a time, TMEM loads double-buffered one chunk ahead
                auto process16 = [&](const uint32_t (&v)[16], int c0) {
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        float4 bb;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(bb.x), "=f"(bb.y), "=f"(bb.z), "=f"(bb.w)
                                     : "r"(sbias + 4u * (uint32_t)(c0 + j)));
                        f[j] = __uint_as_float(v[j]) + bb.x; f[j + 1] = __uint_as_float(v[j + 1]) + bb.y;
                        f[j + 2] = __uint_as_float(v[j + 2]) + bb.z; f[j + 3] = __uint_as_float(v[j + 3]) + bb.w;
                    }
                    if (need_f32) {
                        if (relu) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
                        }
                        const int src0 = c0 & 16;              // position of this chunk inside the 32-wide lane-held slice
                        if (l == 7) {                          // sigma_out on the fp32 activations (mlps.py:265)
#pragma unroll
                            for (int j = 0; j < 16; ++j) sig = fmaf(f[j], __shfl_sync(0xffffffffu, hw0, src0 + j), sig);
                        }
                        if (l == 9) {                          // color_out on the fp32 color_fc activations (mlps.py:273)
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                rgb[0] = fmaf(f[j], __shfl_sync(0xffffffffu, hw0, src0 + j), rgb[0]);
                                rgb[1] = fmaf(f[j], __shfl_sync(0xffffffffu, hw1, src0 + j), rgb[1]);
                                rgb[2] = fmaf(f[j], __shfl_sync(0xffffffffu, hw2, src0 + j), rgb[2]);
                            }
                        }
                        if (want_dbg && l == p.dbg_layer && valid) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) p.dbg[q * 256 + c0 + j] = f[j];
                        }
                    }
                    if (write_act) {
                        uint32_t w[8];
                        if (relu && !need_f32) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) w[j] = pack2_relu<!STASH>(f[2 * j], f[2 * j + 1]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 8; ++j) w[j] = pack2<!STASH>(f[2 * j], f[2 * j + 1]);
                        }
                        st_chunk(act, (c0 >> 3), r, w[0], w[1], w[2], w[3]);
                        st_chunk(act, (c0 >> 3) + 1, r, w[4], w[5], w[6], w[7]);
                    }
                };
                if (!(want_dbg && l == p.dbg_layer)) {
                    // mask slot: layers 0..7 produce h1..h8 (slots 0..7), color_fc produces c (slot 8); feature has no ReLU
                    uint32_t* gmask = (stash_tile && l != 8)
                                          ? reinterpret_cast<uint32_t*>(stash_tile + kStashMask + (size_t)(l == 9 ? 8 : l) * 4096 + (size_t)r * 32)
                                          : nullptr;
                    if (l <= 6) epi_columns<0, STASH>(tmem_row, sbias, act, r, lane, tail, sig, rgb, gmask);
                    else if (l == 7) epi_columns<1, STASH>(tmem_row, sbias, act, r, lane, tail, sig, rgb, gmask);
                    else if (l == 8) epi_columns<2, STASH>(tmem_row, sbias, act, r, lane, tail, sig, rgb, gmask);
                    else epi_columns<3, STASH>(tmem_row, sbias, act, r, lane, tail, sig, rgb, gmask);
                } else {
                uint32_t va[16], vb[16];
                tc_ld16(tmem_row, va);
                for (int c0 = 0; c0 < N; c0 += 32) {
                    tc_wait_ld();
                    pin16(va);
                    tc_ld16(tmem_row + (uint32_t)c0 + 16u, vb);
                    // next 32-wide slice of the head weights (used from the next iteration on)
                    float n0 = 0.f, n1 = 0.f, n2 = 0.f;
                    if (l == 7 && c0 + 32 < N) n0 = __ldg(tail + kWsigOfs + c0 + 32 + lane);
                    if (l == 9 && c0 + 32 < N) {
                        n0 = __ldg(tail + kWoOfs + c0 + 32 + lane); n1 = __ldg(tail + kWoOfs + 128 + c0 + 32 + lane);
                        n2 = __ldg(tail + kWoOfs + 256 + c0 + 32 + lane);
                    }
                    process16(va, c0);
                    tc_wait_ld();
                    pin16(vb);
                    if (c0 + 32 < N) tc_ld16(tmem_row + (uint32_t)c0 + 32u, va);
                    process16(vb, c0 + 16);
                    hw0 = n0; hw1 = n1; hw2 = n2;
                }
                }
                t_cols += clock64() - tc0;
                if (l == 8) {              // gamma(d) for color_fc replaces gamma(x) (layer 4 has retired)
                    if (FROM_ENC) copy_enc_row<!STASH>(gx, r, valid ? p.enc_dir + qc * kDirDim : nullptr, kDirDim, 4, srow(kStashGd));
                    else encode_dir<!STASH>(gx, r, vdir[0], vdir[1], vdir[2], srow(kStashGd));
                }
                if (do_stash) handoff_signal(t);                // l == 9: only the stash copy of c waits for it
                else if (l != 9) { tc_fence_before(); fence_async_smem(); arrive_in(crank, bar_in, bar_pin, t); }
            }
            if (valid) {
                reinterpret_cast<float4*>(p.raw)[q] = make_float4(rgb[0] + tail[kBoOfs], rgb[1] + tail[kBoOfs + 1],
                                                                   rgb[2] + tail[kBoOfs + 2], sig + tail[kBsigOfs]);
            }
            tc_fence_before();   // the next pair's first MMA overwrites this accumulator: order our tcgen05.ld before it
        }
        if (p.cyc && blockIdx.x == 0 && (r == 0)) {
            p.cyc[5 + 4 * t] = (unsigned long long)w_acc; p.cyc[6 + 4 * t] = (unsigned long long)w_bar;
            p.cyc[7 + 4 * t] = (unsigned long long)t_cols; p.cyc[8 + 4 * t] = (unsigned long long)(clock64() - t_begin);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();          // neither CTA leaves (or frees TMEM) while the pair's MMAs or commits may still touch it
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// =======================================================================================================
// fp32-ACCURATE forward on the tensor cores (inference; the eval path of the fp32 parity mode).  Every operand is split into
// two fp16 terms, x = hi + 2^-11 lo with hi = fp16(x), lo = fp16(2^11 (x - hi)) -- the residual is scaled into fp16's NORMAL
// range (unscaled, the residual of a weight of magnitude 0.05 is a subnormal with 2^-21 relative resolution) -- 22 significant
// bits together, and every layer is
//     acc = A_hi W_hi  +  2^-11 (A_hi W_lo + A_lo W_hi)            (the dropped lo*lo term is 2^-22 relative)
// -- three kind::f16 MMAs per K = 16 step: the main term into TMEM columns [0,256), the two cross terms into [256,512); the
// epilogue combines them.  fp16 products are exact in fp32, so what is left against an fp32 FFMA chain is accumulation order
// and that last term.  Same CTA-pair machinery as the kernel above; the second activation
// tile's shared memory holds the LOW halves, so a CTA works on ONE 128-point tile at a time (no ping-pong): the weight ring
// streams a hi and a lo half-slab per K = 32 slab, warps 4-7 own rows and columns [0,128), warps 8-11 the same rows and
// columns [128,256) (both warp groups can read the tile's TMEM lanes), heads as in the kernel above.
// =======================================================================================================
__device__ __forceinline__ float2 f16x2_to_f32(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }
// 8 consecutive K elements of row r -> one 16-byte chunk in the hi image and one in the lo image
template <bool RELU>
__device__ __forceinline__ void st_split8(uint32_t img_hi, uint32_t img_lo, int k8, int r, const float* v) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = RELU ? fmaxf(v[2 * j], 0.f) : v[2 * j], b = RELU ? fmaxf(v[2 * j + 1], 0.f) : v[2 * j + 1];
        hi[j] = pack_f16(a, b);
        const float2 h = f16x2_to_f32(hi[j]);
        lo[j] = pack_f16((a - h.x) * 2048.0f, (b - h.y) * 2048.0f);
    }
    st_chunk(img_hi, k8, r, hi[0], hi[1], hi[2], hi[3]);
    st_chunk(img_lo, k8, r, lo[0], lo[1], lo[2], lo[3]);
}
__device__ __forceinline__ void encode_pos_split(uint32_t gx_hi, uint32_t gx_lo, int r, float px, float py, float pz) {
    float e[64];
    e[0] = px; e[1] = py; e[2] = pz; e[63] = 0.f;
    float s[3], c[3];
    sincosf(px, &s[0], &c[0]); sincosf(py, &s[1], &c[1]); sincosf(pz, &s[2], &c[2]);
#pragma unroll
    for (int k = 0; k < 10; ++k) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            e[3 + 3 * k + d] = s[d]; e[33 + 3 * k + d] = c[d];
            if (k < 9) {      // exact argument doubling would accumulate rounding over 9 octaves at the 1e-4 bar: re-evaluate
                const float a = ldexpf(d == 0 ? px : (d == 1 ? py : pz), k + 1);
                sincosf(a, &s[d], &c[d]);
            }
        }
    }
#pragma unroll
    for (int k8 = 0; k8 < 8; ++k8) st_split8<false>(gx_hi, gx_lo, k8, r, e + 8 * k8);
}
__device__ __forceinline__ void encode_dir_split(uint32_t gx_hi, uint32_t gx_lo, int r, float vx, float vy, float vz) {
    float e[32];
#pragma unroll
    for (int i = 27; i < 32; ++i) e[i] = 0.f;
    e[0] = vx; e[1] = vy; e[2] = vz;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float v3[3] = {ldexpf(vx, k), ldexpf(vy, k), ldexpf(vz, k)};
#pragma unroll
        for (int d = 0; d < 3; ++d) sincosf(v3[d], &e[3 + 3 * k + d], &e[15 + 3 * k + d]);
    }
#pragma unroll
    for (int k8 = 0; k8 < 4; ++k8) st_split8<false>(gx_hi, gx_lo, k8, r, e + 8 * k8);
}
__device__ __forceinline__ void copy_enc_row_split(uint32_t gx_hi, uint32_t gx_lo, int r, const float* __restrict__ src, int n, int chunks) {
    for (int k8 = 0; k8 < chunks; ++k8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (8 * k8 + j < n && src) ? src[8 * k8 + j] : 0.f;
        st_split8<false>(gx_hi, gx_lo, k8, r, v);
    }
}

template <bool FROM_ENC>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) field_fwd_split_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();
    const uint32_t bar_full = sbase + kSmemBar, bar_empty = bar_full + 8 * kStages2, bar_in = bar_empty + 8 * kStages2,
                   bar_acc = bar_in + 16, bar_pin = bar_acc + 16 + 8 * kStages2;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kSmemBar + 8 * (3 * kStages2 + 6));
    const uint32_t act_hi = sbase + kSmemAct, act_lo = act_hi + kActBytes, gx_hi = sbase + kSmemGx, gx_lo = gx_hi + kGxBytes;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages2; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_in, 256); mbar_init(bar_acc, 1); mbar_init(bar_pin, 256);      // both epilogue warp groups arrive
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // one tile per CTA and iteration: the pair covers tiles (2 i, 2 i + 1)
    const int64_t num_pairs = (p.num_tiles + 1) / 2;
    const int64_t first_pair = (int64_t)(blockIdx.x >> 1);
    const int64_t pair_stride = gridDim.x >> 1;
    const int64_t n_iter = first_pair < num_pairs ? (num_pairs - first_pair + pair_stride - 1) / pair_stride : 0;
    const float* tail = reinterpret_cast<const float*>(p.packed + kBiasOfs);

    if (warp == 0) {
        // ---- TMA producer: per K = 32 slab a hi half-slab and a lo half-slab into two consecutive ring stages ----
        uint32_t stage = 0, round = 0;
        for (int64_t it = 0; it < n_iter; ++it) {
            for (int l = 0; l < kNumMmaLayers; ++l) {
                const uint32_t bytes = 32u * (uint32_t)layer_N(l) * 2u, half = bytes >> 1;
                const int ns = layer_nslabs(l);
                for (int s2 = 0; s2 < 2 * ns; ++s2) {
                    const int s = s2 >> 1;
                    const uint32_t img = (s2 & 1) ? kF16LoImgOfs : kF16ImgOfs;
                    mbar_wait(bar_empty + 8 * stage, (round & 1) ^ 1);
                    if (elect_one()) {
                        if (crank == 0) mbar_expect_tx(bar_full + 8 * stage, bytes);
                        tma_load_rows_to_leader(sbase + kSmemRing + stage * kStageBytes2, half == 8192u ? &p.tm8 : &p.tm4,
                                                (img + c_layer_ofs[l] + (uint32_t)s * bytes + crank * half) >> 8, bar_full + 8 * stage);
                    }
                    __syncwarp();
                    if (++stage == kStages2) { stage = 0; ++round; }
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer (leader's elected thread): three MMAs per K = 16 step ----
        if (crank == 0 && elect_one()) {
            uint32_t stage = 0, round = 0, use = 0;
            const uint64_t ahi = desc_hi(2048, 128);
            const uint32_t ring_lo = (sbase + kSmemRing) >> 4;
            for (int64_t it = 0; it < n_iter; ++it) {
                for (int l = 0; l < kNumMmaLayers; ++l, ++use) {
                    const int N = layer_N(l);
                    const uint32_t idesc = make_idesc2(N, kFmtF16, kFmtF16);
                    const uint32_t lbo_b = (uint32_t)N * 8u;
                    const uint64_t bhi = desc_hi(lbo_b, 128);
                    const uint32_t b_step = (2u * lbo_b) >> 4;
                    const int n_act = l == 0 ? 0 : 8;
                    const int n_gx = l == 0 ? 2 : (l == 4 ? 2 : (l == 9 ? 1 : 0));
                    mbar_wait(bar_in, use & 1);
                    mbar_wait_cl(bar_pin, use & 1);
                    tc_fence_after();
                    bool first = true;
                    const uint32_t d_main = tmem_base, d_cross = tmem_base + 256u;
                    for (int seg = 0; seg < 2; ++seg) {
                        const int n = seg == 0 ? n_act : n_gx;
                        uint32_t a_h = (seg == 0 ? act_hi : gx_hi) >> 4, a_l = (seg == 0 ? act_lo : gx_lo) >> 4;
                        for (int s = 0; s < n; ++s, a_h += 512u, a_l += 512u) {
                            const uint32_t st_h = stage, rd = round;
                            if (++stage == kStages2) { stage = 0; ++round; }
                            const uint32_t st_l = stage, rd_l = round;
                            if (++stage == kStages2) { stage = 0; ++round; }
                            mbar_wait(bar_full + 8 * st_h, rd & 1);
                            mbar_wait(bar_full + 8 * st_l, rd_l & 1);
                            tc_fence_after();
                            const uint32_t w_h = ring_lo + st_h * (kStageBytes2 >> 4), w_l = ring_lo + st_l * (kStageBytes2 >> 4);
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const uint32_t ao = (uint32_t)h * 256u, bo = (uint32_t)h * b_step;
                                tc_mma2(d_main, ahi | (uint64_t)(a_h + ao), bhi | (uint64_t)(w_h + bo), idesc, first ? 0u : 1u);
                                tc_mma2(d_cross, ahi | (uint64_t)(a_h + ao), bhi | (uint64_t)(w_l + bo), idesc, first ? 0u : 1u);
                                tc_mma2(d_cross, ahi | (uint64_t)(a_l + ao), bhi | (uint64_t)(w_h + bo), idesc, 1u);
                                first = false;
                            }
                            const bool last = (seg == 1 || n_gx == 0) && s == n - 1;
                            if (last) tc_commit2(bar_acc);
                            tc_commit2(bar_empty + 8 * st_h);
                            tc_commit2(bar_empty + 8 * st_l);
                        }
                    }
                }
            }
        }
    } else if (warp >= 4) {
        // ---- epilogue: thread = (row r, column half g) ----
        const int g = (warp - 4) >> 2;                   // 0: columns [0,128), 1: [128,256)
        const int r = ((warp & 3) << 5) + lane;          // accumulator row == TMEM lane == point within the tile
        const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        float* sbias = reinterpret_cast<float*>(smem + kSmemBias);          // 256 fp32: the current layer's bias
        float* shead = sbias;      // 128 x 4 fp32 (the whole 2 KB block): head partial sums of group 1, after the last layer
        uint32_t use = 0;
        for (int64_t it = 0, pair = first_pair; it < n_iter; ++it, pair += pair_stride) {
            const int64_t tile = pair * 2 + crank;
            const int64_t q = tile * TILE_M + r;
            const bool valid = tile < p.num_tiles && q < p.Q;
            const int64_t qc = valid ? q : 0;
            if (g == 0) {                                // (the encodings are this row's work once: group 0 writes them)
                if (FROM_ENC) {
                    copy_enc_row_split(gx_hi, gx_lo, r, valid ? p.enc_pos + qc * kPosDim : nullptr, kPosDim, 8);
                } else {
                    const int64_t b = qc / p.N;
                    const float zz = valid ? p.z[qc] : 0.f;
                    const float zm = p.ray_norm ? zz * p.ray_norm[b] : zz;
                    encode_pos_split(gx_hi, gx_lo, r, fmaf(p.rays_d[b * 3 + 0], zm, p.rays_o[b * 3 + 0]), fmaf(p.rays_d[b * 3 + 1], zm, p.rays_o[b * 3 + 1]),
                                     fmaf(p.rays_d[b * 3 + 2], zm, p.rays_o[b * 3 + 2]));
                }
            }
            fence_async_smem(); arrive_in(crank, bar_in, bar_pin, 0);
            float sig = 0.f, rgb[3] = {0.f, 0.f, 0.f};
            for (int l = 0; l < kNumMmaLayers; ++l, ++use) {
                const int N = layer_N(l);
                const int c_begin = g * (N >> 1), c_end = c_begin + (N >> 1);
                mbar_wait(bar_acc, use & 1);
                tc_fence_after();
                named_bar_sync(1, 256);                  // everyone is past the previous layer's reads of sbias / shead
                if (threadIdx.x - 128 < (unsigned)N) sbias[threadIdx.x - 128] = __ldg(tail + layer_bias_ofs(l) + (threadIdx.x - 128));
                named_bar_sync(1, 256);
                for (int c0 = c_begin; c0 < c_end; c0 += 16) {
                    uint32_t v[16], vc[16];
                    tc_ld16(tmem_row + (uint32_t)c0, v);
                    tc_ld16(tmem_row + 256u + (uint32_t)c0, vc);
                    tc_wait_ld();
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) f[j] = fmaf(__uint_as_float(vc[j]), 1.0f / 2048.0f, __uint_as_float(v[j])) + sbias[c0 + j];
                    if (l != 8) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
                    }
                    if (l == 7) {                        // sigma_out on the fp32 activations (mlps.py:265)
#pragma unroll
                        for (int j = 0; j < 16; ++j) sig = fmaf(f[j], __ldg(tail + kWsigOfs + c0 + j), sig);
                    }
                    if (l == 9) {                        // color_out on the fp32 color_fc activations (mlps.py:273)
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            rgb[0] = fmaf(f[j], __ldg(tail + kWoOfs + c0 + j), rgb[0]);
                            rgb[1] = fmaf(f[j], __ldg(tail + kWoOfs + 128 + c0 + j), rgb[1]);
                            rgb[2] = fmaf(f[j], __ldg(tail + kWoOfs + 256 + c0 + j), rgb[2]);
                        }
                    }
                    if (p.dbg && l == p.dbg_layer && valid) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) p.dbg[q * 256 + c0 + j] = f[j];
                    }
                    if (l != 9) {                        // next layer's A operand (hi and lo images), in place
                        st_split8<false>(act_hi, act_lo, (c0 >> 3), r, f);
                        st_split8<false>(act_hi, act_lo, (c0 >> 3) + 1, r, f + 8);
                    }
                }
                if (l == 8 && g == 1) {                  // gamma(d) for color_fc replaces gamma(x) (layer 4 has retired)
                    if (FROM_ENC) copy_enc_row_split(gx_hi, gx_lo, r, valid ? p.enc_dir + qc * kDirDim : nullptr, kDirDim, 4);
                    else {
                        const int64_t b = qc / p.N;
                        const float* vs = p.viewdirs ? p.viewdirs : p.rays_d;
                        const float vx = vs[b * 3 + 0], vy = vs[b * 3 + 1], vz = vs[b * 3 + 2];
                        const float inv = 1.0f / fmaxf(sqrtf(vx * vx + vy * vy + vz * vz), 1e-12f);
                        encode_dir_split(gx_hi, gx_lo, r, vx * inv, vy * inv, vz * inv);
                    }
                }
                if (l != 9) { tc_fence_before(); fence_async_smem(); arrive_in(crank, bar_in, bar_pin, 0); }
            }
            // combine the two column halves of the head sums: group 1 hands its partials to group 0 through shared memory
            named_bar_sync(1, 256);
            if (g == 1) { shead[4 * r + 0] = rgb[0]; shead[4 * r + 1] = rgb[1]; shead[4 * r + 2] = rgb[2]; shead[4 * r + 3] = sig; }
            named_bar_sync(1, 256);
            if (g == 0 && valid)
                reinterpret_cast<float4*>(p.raw)[q] = make_float4(rgb[0] + shead[4 * r + 0] + tail[kBoOfs], rgb[1] + shead[4 * r + 1] + tail[kBoOfs + 1],
                                                                   rgb[2] + shead[4 * r + 2] + tail[kBoOfs + 2], sig + shead[4 * r + 3] + tail[kBsigOfs]);
            tc_fence_before();
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ---- weight packing: flat fp32 params -> bf16 shared-memory images + fp32 tail ------------------------
__device__ __forceinline__ float f16_residual(float x) {      // 2^11 (x - fp16(x)): exact in fp32, in fp16's normal range
    const __half h = __float2half_rn(fminf(fmaxf(x, -65504.0f), 65504.0f));
    return (x - __half2float(h)) * 2048.0f;
}
// FMT 0: bf16 image   1: fp16 image (= the high halves of the split)   2: low halves of the split
template <int FMT>
__device__ __forceinline__ void pack_tc_forward(const float* __restrict__ params, uint8_t* __restrict__ out, int m) {
    constexpr bool F16 = FMT != 0;
    // MMA layer m (0..9) <- parameter layer index: 0..7 trunk, 8 feature, 10 color_fc
    {
        const int pl = m < 9 ? m : 10;
        const LayerDesc d = layer_desc(pl);
        const int N = d.N, Kp = d.Kpad;
        __nv_bfloat16* img = reinterpret_cast<__nv_bfloat16*>(out + (FMT == 2 ? kF16LoImgOfs : FMT == 1 ? kF16ImgOfs : 0u) + c_layer_ofs[m]);   // (16-bit elements)
        // image order: [K slab k/32][half of N (one per CTA of a pair)][K chunk (k/8)%4][n % (N/2)][k%8] -- a CTA's half
        // of a K=32 slab is one contiguous block (8 KB at N=256).  One 16-byte chunk (8 consecutive k of one row) per
        // thread, consecutive threads on consecutive rows: sector-sized reads, fully coalesced writes.
        const int hn = N >> 1;
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < N * (Kp >> 3); idx += gridDim.x * blockDim.x) {
            const int k8 = idx / N, n = idx % N;
            const float* row = params + d.w_off + (int64_t)n * d.K + 8 * k8;
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float a = 8 * k8 + 2 * j < d.K ? row[2 * j] : 0.f, b = 8 * k8 + 2 * j + 1 < d.K ? row[2 * j + 1] : 0.f;
                if (FMT == 2) { a = f16_residual(a); b = f16_residual(b); }
                w[j] = pack2<F16>(a, b);
            }
            reinterpret_cast<uint4*>(img)[(((size_t)(k8 >> 2) * 2 + n / hn) * 4 + (k8 & 3)) * hn + n % hn] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (FMT != 0) return;                              // the fp32 tail is written once, by the bf16 pass
        float* tail = reinterpret_cast<float*>(out + kBiasOfs);
        for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x)
            tail[layer_bias_ofs(m) + n] = params[d.b_off + n];
    }
    if (m == 0) {
        float* tail = reinterpret_cast<float*>(out + kBiasOfs);
        const LayerDesc ds = layer_desc(9), dc = layer_desc(11);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 256; i += gridDim.x * blockDim.x) tail[kWsigOfs + i] = params[ds.w_off + i];
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 384; i += gridDim.x * blockDim.x) tail[kWoOfs + i] = params[dc.w_off + i];
        if (blockIdx.x == 0 && threadIdx.x < 4) {
            tail[kBsigOfs + threadIdx.x] = threadIdx.x == 0 ? params[ds.b_off] : 0.f;
            tail[kBoOfs + threadIdx.x] = threadIdx.x < 3 ? params[dc.b_off + threadIdx.x] : 0.f;
        }
    }
}

// =======================================================================================================
// Backward, part 1: the dgrad chain (same machinery as the forward: weights^T streamed by TMA, two tiles per
// CTA, accumulators in TMEM).  d_raw -> dY_9 (color_fc pre-activation grad) -> dY_8 (d feature) -> dY_7 .. dY_0;
// every dY tile is bulk-stored to the gradient stash for the wgrad kernel.  ReLU masks come from the forward
// stash (coalesced 16-byte loads of the bf16 images straight from global memory).
// =======================================================================================================
struct DgradParams {
    const float* d_raw;           // [Q,4]
    const uint8_t* packed;        // transposed images at kTImgOfs; fp32 tail (w_sigma, Wo)
    const uint8_t* stash;         // forward stash
    uint8_t* dstash;              // gradient stash (output)
    int64_t Q; int64_t num_tiles;
    alignas(64) CUtensorMap tm8;  // the packed buffer as rows of 256 B, boxes of 32 rows (one 8 KB half slab)
};

__device__ __forceinline__ uint4 ldg16(const uint8_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// dgrad epilogue column loop.  KIND 0: plain (feature is linear)   1: + d_sigma * w_sigma, then ReLU mask   2: ReLU mask
// The mask comes as 8 bit words per row (one per 32 columns) written by the forward epilogue -- loaded once per layer,
// so nothing inside the column loop waits on global memory.
template <int KIND>
__device__ __forceinline__ void dgrad_chunk16(const uint32_t (&v)[16], int c0, uint32_t act, int r, float dsig, float hw0, uint32_t bits16) {
    uint32_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float a = __uint_as_float(v[2 * j]), b = __uint_as_float(v[2 * j + 1]);
        if (KIND == 1) {
            a = fmaf(dsig, __shfl_sync(0xffffffffu, hw0, (c0 & 16) + 2 * j), a);
            b = fmaf(dsig, __shfl_sync(0xffffffffu, hw0, (c0 & 16) + 2 * j + 1), b);
        }
        w[j] = pack_bf16(a, b);
        if (KIND != 0) w[j] &= relu_mask_word(bits16, j);
    }
    st_chunk(act, (c0 >> 3), r, w[0], w[1], w[2], w[3]);
    st_chunk(act, (c0 >> 3) + 1, r, w[4], w[5], w[6], w[7]);
}
template <int KIND>
__device__ __forceinline__ void dgrad_columns(uint32_t tmem_row, uint32_t act, int r, int lane, const float* __restrict__ tail,
                                              const uint4& mlo, const uint4& mhi, float dsig) {
    float hw0 = KIND == 1 ? __ldg(tail + kWsigOfs + lane) : 0.f;
    const uint32_t mw[8] = {mlo.x, mlo.y, mlo.z, mlo.w, mhi.x, mhi.y, mhi.z, mhi.w};
    uint32_t va[16], vb[16];
    tc_ld16(tmem_row, va);
#pragma unroll
    for (int i = 0; i < 8; ++i) {                 // fully unrolled: mask words are indexed statically
        const int c0 = 32 * i;
        float n0 = 0.f;
        if (KIND == 1 && i < 7) n0 = __ldg(tail + kWsigOfs + c0 + 32 + lane);
        tc_wait_ld();
        tc_ld16(tmem_row + (uint32_t)c0 + 16u, vb);
        pin16(va);
        dgrad_chunk16<KIND>(va, c0, act, r, dsig, hw0, mw[i]);
        tc_wait_ld();
        tc_ld16(tmem_row + (uint32_t)(i < 7 ? c0 + 32 : c0), va);    // last iteration: harmless re-read
        pin16(vb);
        dgrad_chunk16<KIND>(vb, c0 + 16, act, r, dsig, hw0, mw[i] >> 8);
        hw0 = n0;
    }
}

// the dgrad chain has no gamma(x)/gamma(d) operand, so its weight ring takes that space too: 96 KB = 12 half-slab stages;
// it has no bias staging either, so its (larger) barrier block runs into that space
constexpr int kDgStages = 12;
constexpr int kDgSmemRing = kSmemGx;
static_assert(kDgSmemRing + kDgStages * kStageBytes2 == kSmemBar, "dgrad ring must end at the barrier block");
static_assert(kSmemBar + 8 * (3 * kDgStages + 6) + 4 <= kSmemBytes, "barrier block overflow");
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) field_dgrad_kernel(const __grid_constant__ DgradParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();
    // same CTA-pair protocol as the forward kernel: full/in local, empty/acc via the leader's multicast commits, peer_* in the leader
    const uint32_t bar_full = sbase + kSmemBar, bar_empty = bar_full + 8 * kDgStages, bar_in = bar_empty + 8 * kDgStages,
                   bar_acc = bar_in + 16, bar_pfull = bar_acc + 16, bar_pin = bar_pfull + 8 * kDgStages;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kSmemBar + 8 * (3 * kDgStages + 6));
    if (threadIdx.x == 0) {
        for (int s = 0; s < kDgStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); mbar_init(bar_pfull + 8 * s, 1); }
        for (int t = 0; t < 2; ++t) { mbar_init(bar_in + 8 * t, 1); mbar_init(bar_acc + 8 * t, 1); mbar_init(bar_pin + 8 * t, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t num_pairs = (p.num_tiles + 1) / 2;
    const int64_t first_pair = (int64_t)blockIdx.x - crank;       // lockstep: both CTAs of a cluster run the leader's trip count
    const int64_t n_iter = first_pair < num_pairs ? (num_pairs - first_pair + gridDim.x - 1) / gridDim.x : 0;
    const float* tail = reinterpret_cast<const float*>(p.packed + kBiasOfs);

    if (warp == 0) {
        {                                                  // TMA producer: K=32 x N=256 slabs of W^T
            uint32_t stage = 0, round = 0;
            for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
                for (int m = 0; m < kNumDgradLayers; ++m) {
                    const uint8_t* src = p.packed + dgrad_layer_ofs(m);
                    const int ns = m == 0 ? 4 : 8;
                    for (int s = 0; s < ns; ++s) {                 // fetched once per step, used by tile A then tile B
                        mbar_wait(bar_empty + 8 * stage, (round & 1) ^ 1);
                        if (elect_one()) {      // this CTA's half of the slab (input features [128 crank, +128)) -> leader's barrier
                            if (crank == 0) mbar_expect_tx(bar_full + 8 * stage, kStageBytes);
                            tma_load_rows_to_leader(sbase + kDgSmemRing + stage * kStageBytes2, &p.tm8,
                                                    (dgrad_layer_ofs(m) + (uint32_t)s * kStageBytes + crank * kStageBytes2) >> 8, bar_full + 8 * stage);
                        }
                        __syncwarp();
                        if (++stage == kDgStages) { stage = 0; ++round; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (crank == 0 && elect_one()) {                   // MMA issuer: the leader's elected thread, ping-pong over the two tiles
            uint32_t stage = 0, round = 0, use = 0;
            const uint32_t idesc = make_idesc2(256, kFmtBF16, kFmtBF16);
            const uint64_t ahi = desc_hi(2048, 128), bhi = desc_hi(2048, 128);
            const uint32_t ring_lo = (sbase + kDgSmemRing) >> 4;
            for (int64_t it = 0; it < n_iter; ++it) {
                for (int m = 0; m < kNumDgradLayers; ++m, ++use) {
                    const int ns = m == 0 ? 4 : 8;
                    const uint32_t stage0 = stage, round0 = round;
                    for (int t = 0; t < 2; ++t) {
                        mbar_wait(bar_in + 8 * t, use & 1);
                        mbar_wait_cl(bar_pin + 8 * t, use & 1);
                        tc_fence_after();
                        if (t == 1) { stage = stage0; round = round0; }     // tile B reuses the slabs tile A has just used
                        const uint32_t d_tmem = tmem_base + (uint32_t)t * 256u;
                        uint32_t a_lo = (sbase + kSmemAct + t * kActBytes) >> 4;
                        for (int s = 0; s < ns; ++s, a_lo += 512u) {
                            if (t == 0) {
                                mbar_wait(bar_full + 8 * stage, round & 1);
                                tc_fence_after();
                            }
                            const uint32_t b_lo = ring_lo + stage * (kStageBytes2 >> 4);
                            tc_mma2(d_tmem, ahi | (uint64_t)a_lo, bhi | (uint64_t)b_lo, idesc, s > 0 ? 1u : 0u);
                            tc_mma2(d_tmem, ahi | (uint64_t)(a_lo + 256u), bhi | (uint64_t)(b_lo + 256u), idesc, 1u);
                            if (s == ns - 1) tc_commit2(bar_acc + 8 * t);
                            if (t == 1) tc_commit2(bar_empty + 8 * stage);
                            if (++stage == kDgStages) { stage = 0; ++round; }
                        }
                    }
                }
            }
        }
    } else if (warp == 2 || warp == 3) {
        // operand hand-off + gradient-stash write-out, one warp per tile.  Events per pair: e0 = dY_9 (prologue, 32 KB);
        // e1..e9 = output of chain step e-1 = dY_{8-(e-1)} (64 KB); the last one feeds no MMA.  After every event the group
        // gets its "tile may be overwritten" release (the very first write of the kernel is released up front).
        const int t = warp - 2;
        const uint32_t act = sbase + kSmemAct + t * kActBytes;
        named_bar_arrive(1 + t, 160);
        for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
            const int64_t tile = pair * 2 + t;
            uint8_t* ds_tile = tile < p.num_tiles ? p.dstash + (size_t)tile * kDstashTile : nullptr;
            const bool last_pair = it + 1 == n_iter;
            for (int e = 0; e <= kNumDgradLayers; ++e) {
                handoff_wait(t);
                if (lane == 0) {
                    if (e < kNumDgradLayers) arrive_in(crank, bar_in, bar_pin, t);
                    if (ds_tile) {
                        bulk_s2g(ds_tile + (e == 0 ? dstash_ofs(9) : dstash_ofs(8 - (e - 1))), act, e == 0 ? 32768u : 65536u);
                        bulk_commit();
                        bulk_wait_read0();
                    }
                }
                __syncwarp();
                if (!(last_pair && e == kNumDgradLayers)) named_bar_arrive(1 + t, 160);
            }
        }
        if (lane == 0) bulk_wait_all0();
    } else if (warp >= 4) {
        const int t = (warp - 4) >> 2;
        const int r = (int)threadIdx.x - 128 - t * 128;
        const uint32_t act = sbase + kSmemAct + t * kActBytes;
        const uint32_t tmem_row = tmem_base + (uint32_t)t * 256u + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t use = 0;
        for (int64_t it = 0, pair = blockIdx.x; it < n_iter; ++it, pair += gridDim.x) {
            const int64_t tile = pair * 2 + t;
            const int64_t q = tile * TILE_M + r;
            const bool tile_ok = tile < p.num_tiles;
            const bool valid = tile_ok && q < p.Q;
            const uint8_t* st_tile = p.stash + (size_t)(tile_ok ? tile : 0) * kStashTile;
            // ---- prologue: d_raw -> dY_9 = (d_rgb . Wo) * (c > 0)   (color_out dgrad + color_fc ReLU mask) ----
            const float4 d = valid ? __ldg(reinterpret_cast<const float4*>(p.d_raw) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            named_bar_sync(1 + t, 160);            // the previous pair's last dY image has been copied out of the tile
            {
                const uint8_t* mrow = st_tile + kStashMask + (size_t)r * 32;
                const uint4 cbits = ldg16(mrow + 8 * 4096);                    // c mask (slot 8): 128 columns = 4 words
                const uint32_t cw[4] = {cbits.x, cbits.y, cbits.z, cbits.w};
#pragma unroll
                for (int g = 0; g < 4; ++g) {                                  // 32 columns per lane-held slice of Wo
                    const float w0 = __ldg(tail + kWoOfs + 32 * g + lane), w1 = __ldg(tail + kWoOfs + 128 + 32 * g + lane),
                                w2 = __ldg(tail + kWoOfs + 256 + 32 * g + lane);
#pragma unroll
                    for (int c8 = 0; c8 < 4; ++c8) {
                        const uint32_t bits16 = cw[g] >> (8 * (c8 >> 1));          // chunk (c8/2) of this 32-column word
                        uint32_t w[4];
#pragma unroll
                        for (int j2 = 0; j2 < 4; ++j2) {
                            const int s0 = c8 * 8 + 2 * j2;
                            const float ga = d.x * __shfl_sync(0xffffffffu, w0, s0) + d.y * __shfl_sync(0xffffffffu, w1, s0) +
                                             d.z * __shfl_sync(0xffffffffu, w2, s0);
                            const float gb = d.x * __shfl_sync(0xffffffffu, w0, s0 + 1) + d.y * __shfl_sync(0xffffffffu, w1, s0 + 1) +
                                             d.z * __shfl_sync(0xffffffffu, w2, s0 + 1);
                            w[j2] = pack_bf16(ga, gb) & relu_mask_word(bits16, 4 * (c8 & 1) + j2);
                        }
                        st_chunk(act, g * 4 + c8, r, w[0], w[1], w[2], w[3]);
                    }
                }
            }
            handoff_signal(t);
            for (int m = 0; m < kNumDgradLayers; ++m, ++use) {
                // m == 0: no mask (feature is linear).  m >= 1: output is d(h_{9-m}), masked by h_{9-m} > 0 (mask slot 8-m)
                uint4 mlo = make_uint4(0, 0, 0, 0), mhi = mlo;
                if (m >= 1) {
                    const uint8_t* mrow = st_tile + kStashMask + (size_t)(8 - m) * 4096 + (size_t)r * 32;
                    mlo = ldg16(mrow); mhi = ldg16(mrow + 16);
                }
                mbar_wait(bar_acc + 8 * t, use & 1);
                tc_fence_after();
                named_bar_sync(1 + t, 160);        // the tile's previous image (this step's A operand) has been copied out
                if (m == 0) dgrad_columns<0>(tmem_row, act, r, lane, tail, mlo, mhi, d.w);
                else if (m == 1) dgrad_columns<1>(tmem_row, act, r, lane, tail, mlo, mhi, d.w);
                else dgrad_columns<2>(tmem_row, act, r, lane, tail, mlo, mhi, d.w);
                handoff_signal(t);                 // the last step's image feeds no MMA, only the stash copy
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// =======================================================================================================
// Backward, part 2: wgrad (+ bias and head parameter grads).  gW[n, k] = sum_points dY[pt, n] * X[pt, k]: both operands
// are stashed tile images used as MN-major tcgen05 operands (contraction over the 128 points of a tile); fp32
// accumulators stay in TMEM across all tiles a CTA owns and are flushed once with atomics.  CTAs are split over "jobs"
// (layer x operand block) in proportion to the bytes they stream -- the kernel is HBM-bound, so the tile images arrive
// as 32 KB column-half pieces through a 6-slot TMA ring (always two or more pieces in flight per SM) and each MMA group
// (dY half x X half) starts as soon as its two pieces have landed.  The four otherwise idle warps walk the same pieces in
// shared memory for the CUDA-core reductions: bias grads (column sums of dY) and the sigma_out / color_out weight grads
// (d_raw-weighted column sums of the h8 / c images).
// =======================================================================================================
struct WgPiece { uint32_t ofs; uint32_t bytes; int from_stash; int dy_half; int head; };   // dy_half: -1 (X piece) | 0 | 1
struct WgGroup { int a_piece, b_piece, b_piece2, tmem_col, n; };   // A = dY piece (M = 128 features), B = X piece(s) (N = n columns;
                                                                   // b_piece2 >= 0: second half in the next ring slot, N = 256)
enum { HEAD_NONE = 0, HEAD_SIGMA = 1, HEAD_RGB = 2 };
struct WgradJob {
    int n_pieces; WgPiece pieces[4];
    int n_groups; WgGroup groups[4];
    int release_after[4];  // piece i may be released after group release_after[i] (-1: no MMA uses it)
    int halves, xcols;     // flush geometry: M halves x N columns
    int64_t w_dst;         // float offset of gW[0, col0] in the flat grads
    int ldw;               // row stride of gW (K_true)
    int ncols_valid;       // columns actually present (<= xcols)
    int64_t b_dst;         // float offset of the bias grad, or -1
    int64_t head_w_dst, head_b_dst;   // HEAD_SIGMA: g w_sigma[256], g b_sigma;  HEAD_RGB: g Wo[3][128], g bo[3]
    int cta_begin, cta_count;
};
constexpr int kMaxJobs = 16;
struct WgradParams {
    const uint8_t* stash; const uint8_t* dstash; const float* d_raw; float* grads;
    int64_t num_tiles, Q; int num_jobs; int dbg;
    WgradJob jobs[kMaxJobs];
};
constexpr int kWgPiece = 32768;                       // ring slot: one column half of a tile image
constexpr int kWgSlots = 6;
constexpr int kWgSmemBar = kWgSlots * kWgPiece;       // 196608
constexpr int kWgSmemBytes = kWgSmemBar + 256;
constexpr int kWgThreads = 256;                       // warp 0 producer, warp 1 MMA, warp 2 TMEM alloc, warps 4-7 reductions/flush

// MN-major, no-swizzle descriptor for a tile image used with the POINT index as K: SBO = stride between 8-wide
// column groups (2048 B), LBO = stride between 8-point groups (128 B).
__device__ __forceinline__ uint32_t make_idesc_mn(int N) {
    return (1u << 4) | (kFmtBF16 << 7) | (kFmtBF16 << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}

// Column sums of one piece (chunks w4, w4+4, ... of 8 columns; this lane's rows lane, lane+32, ...):
// KIND 0: plain sum into a0;  1: weighted by d_raw.w into a0;  2: weighted by d_raw.{x,y,z} into a0, a1, a2.
template <int KIND>
__device__ __forceinline__ void wg_colsum(const uint8_t* img, int nchunks, int w4, int lane, const float4 (&dr)[4], float (&a0)[4][8],
                                          float (&a1)[4][8], float (&a2)[4][8]) {
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
        const int c8 = w4 + 4 * ii;
        if (c8 < nchunks) {
#pragma unroll
            for (int rg = 0; rg < 4; ++rg) {
                const uint4 v = *reinterpret_cast<const uint4*>(img + (size_t)c8 * 2048 + (size_t)(rg * 32 + lane) * 16);
                const float x[8] = {bf16lo(v.x), bf16hi(v.x), bf16lo(v.y), bf16hi(v.y), bf16lo(v.z), bf16hi(v.z), bf16lo(v.w), bf16hi(v.w)};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (KIND == 0) a0[ii][j] += x[j];
                    else if (KIND == 1) a0[ii][j] = fmaf(dr[rg].w, x[j], a0[ii][j]);
                    else {
                        a0[ii][j] = fmaf(dr[rg].x, x[j], a0[ii][j]); a1[ii][j] = fmaf(dr[rg].y, x[j], a1[ii][j]);
                        a2[ii][j] = fmaf(dr[rg].z, x[j], a2[ii][j]);
                    }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kWgThreads, 1) field_wgrad_kernel(const __grid_constant__ WgradParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_full = sbase + kWgSmemBar, bar_empty = bar_full + 8 * kWgSlots, bar_done = bar_empty + 8 * kWgSlots;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kWgSmemBar + 8 * (2 * kWgSlots + 2));
    int ji = 0;
    for (int j = 0; j < p.num_jobs; ++j)
        if ((int)blockIdx.x >= p.jobs[j].cta_begin && (int)blockIdx.x < p.jobs[j].cta_begin + p.jobs[j].cta_count) ji = j;
    const WgradJob& job = p.jobs[ji];
    const int part = (int)blockIdx.x - job.cta_begin;
    if (threadIdx.x == 0) {
        // every slot release = one tcgen05.commit (or a plain arrive when no MMA reads the piece) + 4 reduction warps
        for (int s = 0; s < kWgSlots; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1 + 4); }
        mbar_init(bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    int64_t my_tiles = 0;
    for (int64_t tile = part; tile < p.num_tiles; tile += job.cta_count) ++my_tiles;

    if (warp == 0) {
        // producer: the tile's pieces in consumption order, each into the next ring slot
        uint32_t slot = 0, round = 0;
        for (int64_t tile = part; tile < p.num_tiles; tile += job.cta_count) {
            for (int i = 0; i < job.n_pieces; ++i) {
                const WgPiece& pc = job.pieces[i];
                // tiles are walked from the LAST one down: dgrad has just written the gradient stash front to back, so its tail (as much
                // as the 126 MB L2 still holds) is read back without going to HBM
                const int64_t pt = p.num_tiles - 1 - tile;
                const uint8_t* src = pc.from_stash ? p.stash + (size_t)pt * kStashTile + pc.ofs : p.dstash + (size_t)pt * kDstashTile + pc.ofs;
                mbar_wait(bar_empty + 8 * slot, (round & 1) ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(bar_full + 8 * slot, pc.bytes);
                    bulk_g2s(sbase + slot * kWgPiece, src, pc.bytes, bar_full + 8 * slot);
                }
                __syncwarp();
                if (++slot == kWgSlots) { slot = 0; ++round; }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {     // MMA issuer: one elected thread
            uint32_t slot = 0, round = 0;
            const uint64_t mnhi = desc_hi(128, 2048);
            bool first = true;
            long long w_full = 0; const long long t_begin = clock64();
            for (int64_t tile = part; tile < p.num_tiles; tile += job.cta_count) {
                uint32_t pslot[4], pround[4];
                for (int i = 0; i < job.n_pieces; ++i) { pslot[i] = slot; pround[i] = round; if (++slot == kWgSlots) { slot = 0; ++round; } }
                uint32_t ready = 0;                    // bit i: piece i's full barrier has been observed
                for (int g = 0; g < job.n_groups; ++g) {
                    const WgGroup& gr = job.groups[g];
                    const long long tw0 = clock64();
                    if (!(ready >> gr.a_piece & 1)) { mbar_wait(bar_full + 8 * pslot[gr.a_piece], pround[gr.a_piece] & 1); ready |= 1u << gr.a_piece; }
                    if (!(ready >> gr.b_piece & 1)) { mbar_wait(bar_full + 8 * pslot[gr.b_piece], pround[gr.b_piece] & 1); ready |= 1u << gr.b_piece; }
                    if (gr.b_piece2 >= 0 && !(ready >> gr.b_piece2 & 1)) {
                        mbar_wait(bar_full + 8 * pslot[gr.b_piece2], pround[gr.b_piece2] & 1); ready |= 1u << gr.b_piece2;
                    }
                    w_full += clock64() - tw0;
                    tc_fence_after();
                    const uint32_t a_lo = (sbase + pslot[gr.a_piece] * kWgPiece) >> 4, b_lo = (sbase + pslot[gr.b_piece] * kWgPiece) >> 4;
                    const uint32_t idesc = make_idesc_mn(gr.n);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)     // K = 16 points per MMA
                        tc_mma(tmem_base + (uint32_t)gr.tmem_col, mnhi | (uint64_t)(a_lo + ks * 16), mnhi | (uint64_t)(b_lo + ks * 16), idesc,
                               (!first || ks > 0) ? 1u : 0u);
                    for (int i = 0; i < job.n_pieces; ++i)
                        if (job.release_after[i] == g) tc_commit(bar_empty + 8 * pslot[i]);
                }
                for (int i = 0; i < job.n_pieces; ++i)      // pieces no MMA reads (head-only jobs): plain arrive
                    if (job.release_after[i] < 0) { mbar_wait(bar_full + 8 * pslot[i], pround[i] & 1); mbar_arrive(bar_empty + 8 * pslot[i]); }
                first = false;
            }
            tc_commit(bar_done);
            if (p.dbg && (part == 0)) printf("wgrad job %d (%d CTAs, %lld tiles): mma thread waited for pieces %lld of %lld cycles\n", ji, job.cta_count, (long long)my_tiles, w_full, clock64() - t_begin);
        }
    } else if (warp >= 4) {
        // ---- CUDA-core reductions over the pieces in shared memory (lanes over points -> conflict-free 16-byte reads) ----
        const int w4 = warp - 4;
        float bsum[2][4][8];            // bias grads: [dY half][chunk w4+4i][8 columns]
        float hacc[3][4][8];            // HEAD_SIGMA: [X half][chunk][8];  HEAD_RGB: [channel][chunk][8] (c = one 128-column piece)
        float dsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) { bsum[0][i][j] = bsum[1][i][j] = 0.f; hacc[0][i][j] = hacc[1][i][j] = hacc[2][i][j] = 0.f; }
        const bool want_bias = job.b_dst >= 0;
        int job_head = HEAD_NONE;
        for (int i = 0; i < job.n_pieces; ++i) if (job.pieces[i].head) job_head = job.pieces[i].head;
        auto load_dr = [&](int64_t tile, float4 (&dr)[4]) {
#pragma unroll
            for (int rg = 0; rg < 4; ++rg) {
                const int64_t q = (p.num_tiles - 1 - tile) * TILE_M + rg * 32 + lane;
                dr[rg] = (tile < p.num_tiles && q < p.Q) ? __ldg(reinterpret_cast<const float4*>(p.d_raw) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        {
            uint32_t slot = 0, round = 0;
            float4 dr[4], dr_next[4];          // d_raw of this lane's four rows, prefetched one tile ahead (head jobs only)
            if (job_head) load_dr(part, dr_next);
            for (int64_t tile = part; tile < p.num_tiles; tile += job.cta_count) {
                if (job_head) {
#pragma unroll
                    for (int rg = 0; rg < 4; ++rg) dr[rg] = dr_next[rg];
                    load_dr(tile + job.cta_count, dr_next);
                    if (w4 == 0) {
#pragma unroll
                        for (int rg = 0; rg < 4; ++rg) { dsum[0] += dr[rg].x; dsum[1] += dr[rg].y; dsum[2] += dr[rg].z; dsum[3] += dr[rg].w; }
                    }
                }
                int xhalf = 0;
                for (int i = 0; i < job.n_pieces; ++i) {
                    const WgPiece& pc = job.pieces[i];
                    mbar_wait(bar_full + 8 * slot, round & 1);      // also paces the arrivals on the ring
                    const uint8_t* img = smem + slot * kWgPiece;
                    const int nchunks = (int)(pc.bytes >> 11);      // 8-column groups in this piece
                    if (pc.dy_half == 0 && want_bias) wg_colsum<0>(img, nchunks, w4, lane, dr, bsum[0], bsum[0], bsum[0]);
                    else if (pc.dy_half == 1 && want_bias) wg_colsum<0>(img, nchunks, w4, lane, dr, bsum[1], bsum[1], bsum[1]);
                    if (pc.head == HEAD_SIGMA) {
                        if (xhalf == 0) wg_colsum<1>(img, nchunks, w4, lane, dr, hacc[0], hacc[0], hacc[0]);
                        else wg_colsum<1>(img, nchunks, w4, lane, dr, hacc[1], hacc[1], hacc[1]);
                        ++xhalf;
                    } else if (pc.head == HEAD_RGB) {
                        wg_colsum<2>(img, nchunks, w4, lane, dr, hacc[0], hacc[1], hacc[2]);
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_empty + 8 * slot);
                    if (++slot == kWgSlots) { slot = 0; ++round; }
                }
            }
        }
        if (my_tiles > 0) {
            if (want_bias) {
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float sum = warp_sum(bsum[a][ii][j]);
                            if (lane == 0 && a < job.halves) atomicAdd(p.grads + job.b_dst + a * 128 + (w4 + 4 * ii) * 8 + j, sum);
                        }
            }
            if (job_head == HEAD_SIGMA) {
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float sum = warp_sum(hacc[a][ii][j]);
                            if (lane == 0) atomicAdd(p.grads + job.head_w_dst + a * 128 + (w4 + 4 * ii) * 8 + j, sum);
                        }
                if (w4 == 0) { const float sd = warp_sum(dsum[3]); if (lane == 0) atomicAdd(p.grads + job.head_b_dst, sd); }
            } else if (job_head == HEAD_RGB) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float sum = warp_sum(hacc[ch][ii][j]);
                            if (lane == 0) atomicAdd(p.grads + job.head_w_dst + ch * 128 + (w4 + 4 * ii) * 8 + j, sum);
                        }
                if (w4 == 0) {
                    const float a0 = warp_sum(dsum[0]), a1 = warp_sum(dsum[1]), a2 = warp_sum(dsum[2]);
                    if (lane == 0) { atomicAdd(p.grads + job.head_b_dst, a0); atomicAdd(p.grads + job.head_b_dst + 1, a1); atomicAdd(p.grads + job.head_b_dst + 2, a2); }
                }
            }
            // ---- flush: TMEM accumulators -> fp32 atomics on the flat gradient ----
            if (job.n_groups > 0) {
                mbar_wait(bar_done, 0);
                tc_fence_after();
                for (int h = 0; h < job.halves; ++h) {
                    const int n = h * 128 + w4 * 32 + lane;                 // output feature (row of gW)
                    const uint32_t trow = tmem_base + (uint32_t)h * 256u + ((uint32_t)(w4 * 32) << 16);
                    for (int c0 = 0; c0 < job.xcols; c0 += 32) {
                        uint32_t v[32];
                        tc_ld32(trow + (uint32_t)c0, v);
                        tc_wait_ld();
                        float* dst = p.grads + job.w_dst + (int64_t)n * job.ldw + c0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c0 + j < job.ncols_valid) atomicAdd(dst + j, __uint_as_float(v[j]));
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// =======================================================================================================
// Backward, part 3 (only when input gradients are asked for): gradients w.r.t. the two encodings from the dY images the dgrad
// chain left in the gradient stash,
//     d gamma(x) = dY_0 . W_0[:, 0:63] + dY_4 . W_4[:, 256:319]      d gamma(d) = dY_9 . W_cfc[:, 256:283]
// One CTA per SM (cta_group::1), persistent over 128-point tiles.  The three B images (72 KB) stay resident in shared memory;
// a tile's A images (dY_0, dY_4: K = 256; dY_9: K = 128; 160 KB) stream through a 4-slot ring of K = 64 slabs (16 KB, one
// contiguous piece of a stash image) by bulk copies.  Both gamma(x) products chain into one N = 64 accumulator, gamma(d) into an
// N = 32 one; two accumulator sets in TMEM, so the epilogue of a tile overlaps the MMAs of the next.  The epilogue (thread =
// point) stages fp32 rows in shared memory and stores them coalesced.  1.25 KB read and 360 B written per point: HBM-bound.
// Roles: warp 0 producer, warp 1 MMA issuer, warp 2 TMEM allocation, warps 4-7 epilogue.
// =======================================================================================================
struct DinputParams {
    const uint8_t* packed; const uint8_t* dstash;
    float* d_enc_pos; float* d_enc_dir;                 // [Q,63] / [Q,27], either may be null
    int64_t Q, num_tiles;
};
constexpr int kDiSlab = 16384;
constexpr int kDiStages = 4;
constexpr int kDiSlabs = 10;                           // per tile: dY_0 x 4, dY_4 x 4, dY_9 x 2
constexpr int kDiSmemRing = kDinImgBytes;
constexpr int kDiSmemOut = kDiSmemRing + kDiStages * kDiSlab;
constexpr int kDiOutFloats = TILE_M * (kPosDim + kDirDim);
constexpr int kDiSmemBar = kDiSmemOut + kDiOutFloats * 4;
constexpr int kDiSmemBytes = kDiSmemBar + 256;
constexpr int kDiThreads = 256;
constexpr uint32_t kDiTmemCols = 256;                  // accumulator set a at columns 128 a: gamma(x) [0, 64), gamma(d) [64, 96)
static_assert(kDiSmemBytes <= 227 * 1024, "dinput shared memory");
__host__ __device__ inline size_t dinput_slab_ofs(int s) {
    return s < 4 ? dstash_ofs(0) + (size_t)s * kDiSlab : (s < 8 ? dstash_ofs(4) + (size_t)(s - 4) * kDiSlab : dstash_ofs(9) + (size_t)(s - 8) * kDiSlab);
}

__global__ void __launch_bounds__(kDiThreads, 1) field_dinput_kernel(const __grid_constant__ DinputParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5;
    const uint32_t bar_full = sbase + kDiSmemBar, bar_empty = bar_full + 8 * kDiStages, bar_acc = bar_empty + 8 * kDiStages,
                   bar_free = bar_acc + 16, bar_b = bar_free + 16;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kDiSmemBar + 8 * (2 * kDiStages + 5));
    if (threadIdx.x == 0) {
        for (int s = 0; s < kDiStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_acc + 8 * a, 1); mbar_init(bar_free + 8 * a, 128); }
        mbar_init(bar_b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(kDiTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {                                 // producer: B images once, then the A slabs of every tile
            mbar_expect_tx(bar_b, kDinImgBytes);
            bulk_g2s(sbase, p.packed + kDinImgOfs, kDinImgBytes, bar_b);
            uint32_t stage = 0, round = 0;
            for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                const uint8_t* ds = p.dstash + (size_t)tile * kDstashTile;
                for (int s = 0; s < kDiSlabs; ++s) {
                    mbar_wait(bar_empty + 8 * stage, (round & 1) ^ 1);
                    mbar_expect_tx(bar_full + 8 * stage, kDiSlab);
                    bulk_g2s(sbase + kDiSmemRing + stage * kDiSlab, ds + dinput_slab_ofs(s), kDiSlab, bar_full + 8 * stage);
                    if (++stage == kDiStages) { stage = 0; ++round; }
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {                                 // MMA issuer
            // kind::f16, D = f32, A = B = bf16, both K-major, M = 128
            constexpr uint32_t idesc_base = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE_M >> 4) << 24);
            constexpr uint32_t idesc_x = idesc_base | ((uint32_t)(64 >> 3) << 17), idesc_d = idesc_base | ((uint32_t)(32 >> 3) << 17);
            const uint64_t ahi = desc_hi(2048, 128), bhi_x = desc_hi(64 * 16, 128), bhi_d = desc_hi(32 * 16, 128);
            mbar_wait(bar_b, 0);
            uint32_t stage = 0, round = 0, it = 0;
            for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
                const uint32_t acc = it & 1;
                mbar_wait(bar_free + 8 * acc, ((it >> 1) & 1) ^ 1);          // the epilogue has drained this accumulator set
                tc_fence_after();
                const uint32_t d_x = tmem_base + acc * 128, d_d = d_x + 64;
                for (int s = 0; s < kDiSlabs; ++s) {
                    mbar_wait(bar_full + 8 * stage, round & 1);
                    tc_fence_after();
                    const uint32_t a0 = sbase + kDiSmemRing + stage * kDiSlab;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {                            // K = 16 steps of the slab
                        const uint64_t ad = desc_at(ahi, a0 + j * 4096);
                        if (s < 8) {
                            const uint32_t k0 = (uint32_t)(s & 3) * 64 + j * 16;
                            const uint32_t b = sbase + (s < 4 ? kDinPos0 : kDinPos4) + (k0 >> 3) * 1024;
                            tc_mma(d_x, ad, desc_at(bhi_x, b), idesc_x, (s == 0 && j == 0) ? 0u : 1u);
                        } else {
                            const uint32_t k0 = (uint32_t)(s - 8) * 64 + j * 16;
                            tc_mma(d_d, ad, desc_at(bhi_d, sbase + kDinDir + (k0 >> 3) * 512), idesc_d, (s == 8 && j == 0) ? 0u : 1u);
                        }
                    }
                    tc_commit(bar_empty + 8 * stage);
                    if (++stage == kDiStages) { stage = 0; ++round; }
                }
                tc_commit(bar_acc + 8 * acc);
            }
        }
    } else if (warp >= 4) {
        // epilogue: thread = accumulator row = point of the tile; rows staged in shared memory as the global [rows][63] / [rows][27]
        // blocks (odd row strides: conflict-free), then copied out with consecutive threads on consecutive floats
        const int r = (int)threadIdx.x - 128;
        float* out_x = reinterpret_cast<float*>(smem + kDiSmemOut);
        float* out_d = out_x + TILE_M * kPosDim;
        uint32_t it = 0;
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const uint32_t acc = it & 1;
            mbar_wait(bar_acc + 8 * acc, (it >> 1) & 1);
            tc_fence_after();
            const uint32_t trow = tmem_base + acc * 128 + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
            for (int c = 0; c < 6; ++c) {                                    // columns [0, 64) gamma(x), [64, 96) gamma(d)
                uint32_t v[16];
                tc_ld16(trow + 16 * c, v);
                tc_wait_ld();
                pin16(v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int col = 16 * c + j;
                    if (col < kPosDim) out_x[r * kPosDim + col] = __uint_as_float(v[j]);
                    else if (col >= 64 && col < 64 + kDirDim) out_d[r * kDirDim + col - 64] = __uint_as_float(v[j]);
                }
            }
            tc_fence_before();
            mbar_arrive(bar_free + 8 * acc);
            named_bar_sync(1, 128);
            const int64_t rows = p.Q - tile * TILE_M < TILE_M ? p.Q - tile * TILE_M : TILE_M;
            if (p.d_enc_pos) {
                float* dst = p.d_enc_pos + tile * TILE_M * kPosDim;
                for (int i = r; i < rows * kPosDim; i += 128) dst[i] = out_x[i];
            }
            if (p.d_enc_dir) {
                float* dst = p.d_enc_dir + tile * TILE_M * kDirDim;
                for (int i = r; i < rows * kDirDim; i += 128) dst[i] = out_d[i];
            }
            named_bar_sync(1, 128);                                          // staging area free for the next tile
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kDiTmemCols) : "memory");
    }
}

// B images of field_dinput_kernel: one thread per 16-byte row chunk (8 consecutive out features k of one in feature n)
__device__ __forceinline__ void pack_tc_dinput(const float* __restrict__ params, uint8_t* __restrict__ out) {
    const LayerDesc d0 = layer_desc(0), d4 = layer_desc(4), dc = layer_desc(10);
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * 32 * 64 + 16 * 32; idx += gridDim.x * blockDim.x) {
        int img = idx >> 11, rem = idx & 2047;
        if (img > 2) img = 2;
        if (img == 2) rem = idx - 2 * 2048;
        const int rows = img < 2 ? 64 : 32, n = rem % rows, k8 = rem / rows;
        const LayerDesc& d = img == 0 ? d0 : (img == 1 ? d4 : dc);
        const int col = img == 0 ? n : kHidden + n, n_true = img < 2 ? kPosDim : kDirDim;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = n < n_true ? params[d.w_off + (int64_t)(8 * k8 + j) * d.K + col] : 0.f;
        const uint32_t base = img == 0 ? kDinPos0 : (img == 1 ? kDinPos4 : kDinDir);
        *reinterpret_cast<uint4*>(out + kDinImgOfs + base + (size_t)(k8 * rows + n) * 16) =
            make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
    }
}

// transposed images for the dgrad chain
__device__ __forceinline__ void pack_tc_transposed(const float* __restrict__ params, uint8_t* __restrict__ out, int m) {
    {
        const int pl = m == 0 ? 10 : (m == 1 ? 8 : 9 - m);
        const LayerDesc d = layer_desc(pl);
        const int Nout = d.N;                                  // contraction length (128 or 256)
        __nv_bfloat16* img = reinterpret_cast<__nv_bfloat16*>(out + dgrad_layer_ofs(m));
        // W[n, j], j < 256 <= K; same half-slab order with (k, n) := (n, j); one chunk = 8 consecutive out-features n of one
        // in-feature j per thread, consecutive threads on consecutive j (coalesced reads of 8 rows, coalesced writes)
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < (Nout >> 3) * 256; idx += gridDim.x * blockDim.x) {
            const int n8 = idx >> 8, j = idx & 255;
            const float* col = params + d.w_off + (int64_t)(8 * n8) * d.K + j;
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) w[q] = pack_bf16(col[(int64_t)(2 * q) * d.K], col[(int64_t)(2 * q + 1) * d.K]);
            reinterpret_cast<uint4*>(img)[(((size_t)(n8 >> 2) * 2 + (j >> 7)) * 4 + (n8 & 3)) * 128 + (j & 127)] = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
}
// one launch packs every image of up to four nets: blockIdx.y = forward layer 0..9 (bf16) | 10 + dgrad step 0..8 |
// 19 input-gradient images | 20 + forward layer 0..9 (fp16 = split high halves) | 30 + forward layer 0..9 (split low halves),
// blockIdx.z = net
struct PackBatch { const float* params[4]; uint8_t* out[4]; uint64_t* counter; };
__global__ void pack_tc_kernel(const PackBatch b) {
    // last kernel of a replayed training step: bump the device-side step counter (nothing else in this launch reads it, every
    // reader of the next replay starts after this kernel)
    if (b.counter && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) *b.counter += 1;
    const float* params = b.params[blockIdx.z];
    uint8_t* out = b.out[blockIdx.z];
    if (blockIdx.y < kNumMmaLayers) pack_tc_forward<0>(params, out, blockIdx.y);
    else if (blockIdx.y < kNumMmaLayers + kNumDgradLayers) pack_tc_transposed(params, out, blockIdx.y - kNumMmaLayers);
    else if (blockIdx.y == kNumMmaLayers + kNumDgradLayers) pack_tc_dinput(params, out);
    else if (blockIdx.y < 2 * kNumMmaLayers + kNumDgradLayers + 1) pack_tc_forward<1>(params, out, blockIdx.y - kNumMmaLayers - kNumDgradLayers - 1);
    else pack_tc_forward<2>(params, out, blockIdx.y - 2 * kNumMmaLayers - kNumDgradLayers - 1);
}

}  // namespace tc

size_t tc_packed_bytes() { return align_up(tc::kPackedTcBytes, 256); }

size_t tc_workspace_bytes(int64_t Q, int stash) {
    const int64_t tiles = cdiv(Q, tc::TILE_M);
    return 256 + (stash ? (size_t)tiles * (tc::kStashTile + tc::kDstashTile) : 0);
}
size_t tc_stash_tile_bytes() { return tc::kStashTile; }      // a field workspace offset by k of these starts at tile k
static inline uint8_t* ws_stash(void* ws) { return reinterpret_cast<uint8_t*>(ws) + 256; }
static inline uint8_t* ws_dstash(void* ws, int64_t Q) { return ws_stash(ws) + (size_t)cdiv(Q, tc::TILE_M) * tc::kStashTile; }

int tc_pack(const float* const* params, void* const* packed_bf16, int n_nets, bool train_only, cudaStream_t st) {
    tc::PackBatch b{};
    for (int i = 0; i < n_nets; ++i) { b.params[i] = params[i]; b.out[i] = reinterpret_cast<uint8_t*>(packed_bf16[i]); }
    b.counter = g_pack_counter;
    // blockIdx.y: [0,20) = the training images (bf16 forward + transposed + input-gradient), [20,40) = the inference-only fp16 hi / lo
    const int ny = train_only ? tc::kNumMmaLayers + tc::kNumDgradLayers + 1 : 3 * tc::kNumMmaLayers + tc::kNumDgradLayers + 1;
    tc::pack_tc_kernel<<<dim3(32, ny, n_nets), 256, 0, st>>>(b);
    NSB_LAUNCH_CHECK("pack_tc_kernel");
    return NSB_OK;
}

int check_arch() {
    static int ok = -1;
    if (ok < 0) {
        int dev = 0, major = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
        ok = major == 10 ? 1 : 0;
    }
    return ok ? NSB_OK : NSB_E_ARCH;
}

// ---- tensor maps over a packed-weight buffer (rows of 256 B; boxes of 32 / 16 rows), cached per buffer address ----
struct PackedMaps { const void* ptr; CUtensorMap tm8, tm4; };
static int packed_maps(const void* packed, CUtensorMap* tm8, CUtensorMap* tm4) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static std::mutex mu;
    static EncodeFn encode = nullptr;
    static PackedMaps cache[16];
    static int n_cached = 0, next = 0;
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < n_cached; ++i)
        if (cache[i].ptr == packed) { *tm8 = cache[i].tm8; if (tm4) *tm4 = cache[i].tm4; return NSB_OK; }
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn)
            return check_launch("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled)");
        encode = reinterpret_cast<EncodeFn>(fn);
    }
    PackedMaps m{};
    m.ptr = packed;
    const cuuint64_t dims[2] = {256, tc::kPackedTcBytes / 256};
    const cuuint64_t strides[1] = {256};
    const cuuint32_t estr[2] = {1, 1};
    for (int k = 0; k < 2; ++k) {
        const cuuint32_t box[2] = {256, k == 0 ? 32u : 16u};
        if (encode(k == 0 ? &m.tm8 : &m.tm4, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(packed), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
            snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled failed for the packed weight buffer");
            return NSB_E_CUDA;
        }
    }
    cache[next] = m; next = (next + 1) % 16; if (n_cached < 16) ++n_cached;
    *tm8 = m.tm8; if (tm4) *tm4 = m.tm4;
    return NSB_OK;
}

template <bool FROM_ENC>
static int launch_fwd(tc::FwdParams& p, cudaStream_t st) {
    NSB_TRY(check_arch());
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(tc::field_fwd_kernel<FROM_ENC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(tc::field_fwd_kernel<FROM_ENC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBytes) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(field_fwd_kernel)");
        attr_set = true;
    }
    p.num_tiles = cdiv(p.Q, tc::TILE_M);
    NSB_TRY(packed_maps(p.packed, &p.tm8, &p.tm4));
    const int64_t pairs = (p.num_tiles + 1) / 2;
    int grid = (int)(pairs < num_sms() ? pairs : num_sms());
    grid = (grid + 1) / 2 * 2;                       // clusters of two CTAs (a CTA without a pair idles along)
    if (grid > num_sms()) grid -= 2;
    if (p.stash) tc::field_fwd_kernel<FROM_ENC, true><<<grid, tc::kThreads, tc::kSmemBytes, st>>>(p);
    else tc::field_fwd_kernel<FROM_ENC, false><<<grid, tc::kThreads, tc::kSmemBytes, st>>>(p);
    NSB_LAUNCH_CHECK("field_fwd_kernel");
    return NSB_OK;
}

template <bool FROM_ENC>
static int launch_fwd_split(tc::FwdParams& p, cudaStream_t st) {
    NSB_TRY(check_arch());
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(tc::field_fwd_split_kernel<FROM_ENC>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBytes) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(field_fwd_split_kernel)");
        attr_set = true;
    }
    p.num_tiles = cdiv(p.Q, tc::TILE_M);
    NSB_TRY(packed_maps(p.packed, &p.tm8, &p.tm4));
    const int64_t pairs = (p.num_tiles + 1) / 2;              // a CTA pair takes two tiles per iteration (one per CTA)
    const int64_t max_pairs = num_sms() / 2;
    const int grid = 2 * (int)(pairs < max_pairs ? pairs : max_pairs);
    tc::field_fwd_split_kernel<FROM_ENC><<<grid, tc::kThreads, tc::kSmemBytes, st>>>(p);
    NSB_LAUNCH_CHECK("field_fwd_split_kernel");
    return NSB_OK;
}

// fp32-accurate forward on the tensor cores (fp16 split operands): the inference path of the fp32 parity mode
int tc_field_fwd_rays_split(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm, const float* viewdirs,
                            const void* packed, float* raw, int64_t B, int N, cudaStream_t st) {
    tc::FwdParams p{};
    p.rays_o = rays_o; p.rays_d = rays_d; p.z = z; p.ray_norm = ray_norm; p.viewdirs = viewdirs;
    p.packed = reinterpret_cast<const uint8_t*>(packed); p.raw = raw;
    p.Q = B * (int64_t)N; p.N = N;
    return launch_fwd_split<false>(p, st);
}
int tc_field_fwd_enc_split(const float* enc_pos, const float* enc_dir, const void* packed, float* raw, int64_t Q, cudaStream_t st) {
    tc::FwdParams p{};
    p.enc_pos = enc_pos; p.enc_dir = enc_dir;
    p.packed = reinterpret_cast<const uint8_t*>(packed); p.raw = raw;
    p.Q = Q; p.N = 1;
    return launch_fwd_split<true>(p, st);
}

int tc_field_fwd_rays(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm, const float* viewdirs,
                      const void* packed, float* raw, void* ws, int64_t B, int N, int stash, cudaStream_t st) {
    tc::FwdParams p{};
    p.rays_o = rays_o; p.rays_d = rays_d; p.z = z; p.ray_norm = ray_norm; p.viewdirs = viewdirs;
    p.packed = reinterpret_cast<const uint8_t*>(packed); p.raw = raw;
    p.stash = stash ? ws_stash(ws) : nullptr;
    p.Q = B * (int64_t)N; p.N = N;
    return launch_fwd<false>(p, st);
}

int tc_field_fwd_enc(const float* enc_pos, const float* enc_dir, const void* packed, float* raw, void* ws, int64_t Q,
                     int stash, cudaStream_t st) {
    tc::FwdParams p{};
    p.enc_pos = enc_pos; p.enc_dir = enc_dir;
    p.packed = reinterpret_cast<const uint8_t*>(packed); p.raw = raw;
    p.stash = stash ? ws_stash(ws) : nullptr;
    p.Q = Q; p.N = 1;
    return launch_fwd<true>(p, st);
}

// parameter grads (accumulated into the flat `grads`; none when it is null) and encoding grads (d_enc_pos / d_enc_dir, optional)
// from the forward stash in ws: dgrad chain -> input-gradient products -> wgrad -> head grads
int tc_field_bwd(const float* d_raw, const void* packed, float* grads, float* d_enc_pos, float* d_enc_dir, void* ws, int64_t Q,
                 cudaStream_t st) {
    NSB_TRY(check_arch());
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(tc::field_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(tc::field_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kWgSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(tc::field_dinput_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kDiSmemBytes) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(bwd kernels)");
        attr_set = true;
    }
    const int64_t tiles = cdiv(Q, tc::TILE_M);
    const int64_t pairs = (tiles + 1) / 2;
    tc::DgradParams dp{};
    dp.d_raw = d_raw; dp.packed = reinterpret_cast<const uint8_t*>(packed); dp.stash = ws_stash(ws); dp.dstash = ws_dstash(ws, Q);
    dp.Q = Q; dp.num_tiles = tiles;
    NSB_TRY(packed_maps(packed, &dp.tm8, nullptr));
    int dgrid = (int)(pairs < num_sms() ? pairs : num_sms());
    dgrid = (dgrid + 1) / 2 * 2;                     // clusters of two CTAs
    if (dgrid > num_sms()) dgrid -= 2;
    tc::field_dgrad_kernel<<<dgrid, tc::kThreads, tc::kSmemBytes, st>>>(dp);
    NSB_LAUNCH_CHECK("field_dgrad_kernel");
    if (d_enc_pos || d_enc_dir) {
        tc::DinputParams ip{};
        ip.packed = reinterpret_cast<const uint8_t*>(packed); ip.dstash = ws_dstash(ws, Q);
        ip.d_enc_pos = d_enc_pos; ip.d_enc_dir = d_enc_dir; ip.Q = Q; ip.num_tiles = tiles;
        const int igrid = (int)(tiles < num_sms() ? tiles : num_sms());
        tc::field_dinput_kernel<<<igrid, tc::kDiThreads, tc::kDiSmemBytes, st>>>(ip);
        NSB_LAUNCH_CHECK("field_dinput_kernel");
    }
    if (!grads) return NSB_OK;

    tc::WgradParams wp{};
    wp.stash = ws_stash(ws); wp.dstash = ws_dstash(ws, Q); wp.d_raw = d_raw; wp.grads = grads; wp.num_tiles = tiles; wp.Q = Q;
    int nj = 0;
    // one job = gW block (dY_k columns) x (X block); pieces are 32 KB column halves in consumption order
    auto add = [&](int k, size_t x_ofs, int xcols, int pl, int col0, int valid, bool bias, int head) {
        const LayerDesc d = layer_desc(pl);
        tc::WgradJob& j = wp.jobs[nj++];
        j = tc::WgradJob{};
        const int halves = k == 9 ? 1 : 2;
        const uint32_t dy = (uint32_t)tc::dstash_ofs(k);
        const uint32_t xb = (uint32_t)xcols * 256u;                 // bytes of the X block (xcols/8 chunks x 2048)
        auto piece = [&](uint32_t ofs, uint32_t bytes, int from_stash, int dy_half, int hd) {
            j.pieces[j.n_pieces] = tc::WgPiece{ofs, bytes, from_stash, dy_half, hd}; j.release_after[j.n_pieces] = -1; return j.n_pieces++;
        };
        auto group = [&](int a, int b, int col, int n) {
            j.groups[j.n_groups] = tc::WgGroup{a, b, -1, col, n}; j.release_after[a] = j.n_groups; j.release_after[b] = j.n_groups; ++j.n_groups;
        };
        if (xcols == 256) {
            // X halves first, in adjacent ring slots (a tile takes 4 or 3 of the 6 slots, so the pair starts on slot 0, 2, 4 or 0, 3
            // and never wraps): one N = 256 MMA reads both.  An MN-major MMA costs ~200-250 cycles whatever its N (measured), so
            // halving the instruction count is what counts here.
            const int b0 = piece((uint32_t)x_ofs, 32768, 1, -1, head), b1 = piece((uint32_t)x_ofs + 32768, 32768, 1, -1, head);
            const int a0 = piece(dy, 32768, 0, 0, 0);
            group(a0, b0, 0, 256);
            if (halves == 2) { const int a1 = piece(dy + 32768, 32768, 0, 1, 0); group(a1, b0, 256, 256); }
            for (int g = 0; g < j.n_groups; ++g) j.groups[g].b_piece2 = b1;
            j.release_after[b1] = j.n_groups - 1;
        } else {
            const int a0 = piece(dy, 32768, 0, 0, 0);
            const int b0 = piece((uint32_t)x_ofs, xb, 1, -1, head);
            group(a0, b0, 0, xcols);
            if (halves == 2) { const int a1 = piece(dy + 32768, 32768, 0, 1, 0); group(a1, b0, 256, xcols); }
        }
        j.halves = halves; j.xcols = xcols;
        j.w_dst = d.w_off + col0; j.ldw = d.K; j.ncols_valid = valid; j.b_dst = bias ? d.b_off : -1;
        if (head == tc::HEAD_SIGMA) { const LayerDesc ds = layer_desc(9); j.head_w_dst = ds.w_off; j.head_b_dst = ds.b_off; }
    };
    add(0, tc::kStashGx, 64, 0, 0, 63, true, 0);
    for (int l = 1; l <= 7; ++l) {
        add(l, tc::kStashH + (size_t)(l - 1) * 65536, 256, l, 0, 256, true, 0);
        if (l == 4) add(4, tc::kStashGx, 64, 4, 256, 63, false, 0);
    }
    add(8, tc::kStashH + 7 * 65536, 256, 8, 0, 256, true, tc::HEAD_SIGMA);      // feature; its X = h8 also feeds g w_sigma
    add(9, tc::kStashFeat, 256, 10, 0, 256, true, 0);                           // color_fc [feat | .]
    add(9, tc::kStashGd, 32, 10, 256, 27, false, 0);                            // color_fc [. | gamma(d)]
    {   // color_out: g Wo = d_rgb^T c, g bo -- CUDA-core job over the c image, no MMA
        tc::WgradJob& j = wp.jobs[nj++];
        j = tc::WgradJob{};
        j.pieces[0] = tc::WgPiece{(uint32_t)tc::kStashC, 32768, 1, -1, tc::HEAD_RGB}; j.release_after[0] = -1; j.n_pieces = 1;
        const LayerDesc dc = layer_desc(11);
        j.head_w_dst = dc.w_off; j.head_b_dst = dc.b_off; j.b_dst = -1;
    }
    wp.num_jobs = nj;
    wp.dbg = getenv("NSB_WG_DBG") != nullptr;
    // CTAs per job: greedy min-max of (tiles per CTA) x (cycles per tile).  The per-tile cost is what the MMA thread of
    // each job kind was measured to take on B200 (scripts/perf_bwd.py with NSB_WG_DBG=1): an MN-major MMA costs
    // ~200-250 cycles whatever its N, so cost follows the instruction count more than the bytes.
    const int total = num_sms();
    double cost[tc::kMaxJobs];
    for (int i = 0; i < nj; ++i) {
        const tc::WgradJob& j = wp.jobs[i];
        if (j.n_groups == 0) cost[i] = 1750;                                   // color_out grads, CUDA cores only
        else if (j.xcols == 256) cost[i] = j.halves == 2 ? 5600 : 3100;        // 16 / 8 MMAs of N = 256
        else cost[i] = j.xcols == 64 ? 3750 : 2100;                            // gamma(x) blocks (16 MMAs) / gamma(d) block (8)
        if (j.head_w_dst && j.n_groups) cost[i] += 100;                        // + sigma_out reductions on the idle warps
        wp.jobs[i].cta_count = 1;
    }
    for (int used = nj; used < total; ++used) {
        int worst = -1; double worst_t = -1;
        for (int i = 0; i < nj; ++i) {
            if ((int64_t)wp.jobs[i].cta_count >= tiles) continue;
            const double t = cost[i] * (double)cdiv(tiles, wp.jobs[i].cta_count);
            if (t > worst_t) { worst_t = t; worst = i; }
        }
        if (worst < 0) break;
        ++wp.jobs[worst].cta_count;
    }
    int begin = 0;
    for (int i = 0; i < nj; ++i) { wp.jobs[i].cta_begin = begin; begin += wp.jobs[i].cta_count; }
    tc::field_wgrad_kernel<<<begin, tc::kWgThreads, tc::kWgSmemBytes, st>>>(wp);
    NSB_LAUNCH_CHECK("field_wgrad_kernel");
    return NSB_OK;
}

// debug hook used by tests: run the forward and dump the fp32 post-activation of one layer
int tc_debug_layer(const float* rays_o, const float* rays_d, const float* z, const float* ray_norm, const float* viewdirs,
                   const void* packed, float* raw, float* dbg, int layer, int64_t B, int N, cudaStream_t st) {
    tc::FwdParams p{};
    if (layer < 0) {   // layer -1: cycle counters instead; layer -2: same with the training stash written behind the 32 counters
        p.cyc = reinterpret_cast<unsigned long long*>(dbg);
        if (layer == -2) p.stash = reinterpret_cast<uint8_t*>(dbg) + 256;
        dbg = nullptr;
    }
    p.rays_o = rays_o; p.rays_d = rays_d; p.z = z; p.ray_norm = ray_norm; p.viewdirs = viewdirs;
    p.packed = reinterpret_cast<const uint8_t*>(packed); p.raw = raw; p.dbg = dbg; p.dbg_layer = layer;
    p.Q = B * (int64_t)N; p.N = N;
    return launch_fwd<false>(p, st);
}

}  // namespace nsb
