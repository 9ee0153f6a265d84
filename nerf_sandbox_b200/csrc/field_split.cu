// K1 (fp32 mode, training) -- the layer GEMMs of the fp32 parity mode on the tensor cores.
//
// The fp32 mode keeps every activation and gradient in HBM as fp32 (field_fp32.cu: concat-free buffers, one GEMM per layer
// and role).  This file runs those GEMMs on tcgen05 without giving up fp32 accuracy: each fp32 operand element is split on
// the fly into three bf16 terms  x = x0 + x1 + x2  (x0 = bf16(x), x1 = bf16(x - x0), ...; bf16 keeps fp32's exponent, so
// activations, weights and the tiny back-propagated gradients all split without scaling), and the product is the sum of the
// six term products with i + j < 3, accumulated in fp32 in TMEM: x0 * y0 in one accumulator, the cross products in a second
// one (see the MMA loop for why).  Three terms carry 24 significand bits per operand -- all of an fp32 operand.
//
// One CTA = one 128 x BN output tile (BN = 128 for forward / dgrad with two CTAs per SM, 256 for wgrad with one): 256
// converter threads, an MMA warp and a producer warp.  Per K = 16 chunk every converter thread owns one 8-element piece of
// the fp32 A tile and one (two for BN = 256) of the B tile: cp.async brings it into a thread-private shared-memory slot
// (three chunks in flight per CTA, no registers held, no barrier), the thread splits it and writes the bf16 term images
// into a shared-memory stage in the canonical K-major core-matrix layout -- operands stored with the OTHER index
// contiguous (dgrad's weights, both wgrad operands) are transposed by the same pass, so every MMA is K-major (an MN-major
// MMA costs 3-4x more, DESIGN section 4).  The MMA warp issues the products of a chunk once all its pieces are written
// (mbarrier) and commits them to the stage's "empty" barrier; the stage is rewritten only after that commit has arrived.
// Forward and dgrad take B from term images of the weights written once per optimiser step (split_pack_kernel): the
// producer warp bulk-copies them straight into the stage.  Epilogues by role -- bias + ReLU; addend + mask;
// split-K atomics, plus the bias gradient (column sums of wgrad's A pieces) -- staged through shared memory so that global
// memory sees whole 512-byte rows.  What bounds it is shared-memory bandwidth (DESIGN section 2), not the tensor cores.
#include <cuda_bf16.h>
#include "nsb_common.cuh"
#include "tc_ptx.cuh"

namespace nsb {
namespace tc {

constexpr int SG_BM = 128, SG_BK = 16;                                // output rows per CTA; one K = 16 MMA step per chunk
// output columns per CTA (BN): 128 with two CTAs per SM (forward, dgrad: frequent epilogues overlap the other CTA's main loop),
// 256 with one CTA per SM for wgrad (long contraction, rare epilogue): the A pieces are converted once for both column halves
// and each MMA reads A once for 256 columns -- 1.8x less shared-memory traffic per FLOP
constexpr int SG_CONV = 256;                                          // converter threads = pieces per operand chunk: 128 rows x 2 groups of 8 k
constexpr int SG_THREADS = SG_CONV + 64;                              // + the MMA warp + the weight-image producer warp
constexpr int SG_TERM_BYTES = SG_BM * SG_BK * 2;                      // one bf16 term image of a 128 x 16 operand chunk: [k/8][row][8]
constexpr int SG_RAW_BYTES = SG_BM * SG_BK * 4;                       // the same chunk as fp32
constexpr int SG_FIFO = 4;                                            // raw chunks in flight per CTA (cp.async groups)
constexpr int SG_TERMS = 3;                                           // bf16 terms per fp32 operand element (operands and weight images)
constexpr int SG_IMG_CHUNK = SG_TERMS * SG_TERM_BYTES;                // 12 KB per (128-row tile, K = 16 chunk)
// TMEM: two fp32 accumulators of BN columns: main (x0 * y0) and cross (every other term product)

template <int BN> struct SgCfg {
    static constexpr int kBTiles = BN / 128;                              // B is handled as 128-row operand chunks
    static constexpr int kStageBytes = (1 + kBTiles) * SG_TERMS * SG_TERM_BYTES;   // converted stage: A terms, then B terms ([term][k/8][BN rows][8])
    static constexpr int kStages = 2;
    static constexpr int kFifoOfs = kStages * kStageBytes;
    static constexpr int kFifoSlot = (1 + kBTiles) * SG_RAW_BYTES;        // raw chunk: A, then B
    static constexpr int kBarOfs = kFifoOfs + SG_FIFO * kFifoSlot;
    static constexpr int kEpiLd = BN + 4;                                 // row stride (floats) of the epilogue's shared-memory tile
    static_assert(kBarOfs >= SG_BM * kEpiLd * 4, "the epilogue tile reuses the stage + FIFO area");
    static constexpr int kSmemBytes = kBarOfs + 128;                      // + barriers and the TMEM slot: 112.1 KB (BN 128) / 168.1 KB (BN 256)
    static constexpr uint32_t kTmemCols = 2 * BN;
};

__device__ __forceinline__ uint32_t pack_bf16_pair(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// x[0..8) -> SG_TERMS bf16 term vectors (16 bytes each); the residual of each step is exact in fp32
__device__ __forceinline__ void split8(float (&x)[8], uint4 (&out)[SG_TERMS]) {
#pragma unroll
    for (int t = 0; t < SG_TERMS; ++t) {
        uint32_t p[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) p[j] = pack_bf16_pair(x[2 * j], x[2 * j + 1]);
        out[t] = make_uint4(p[0], p[1], p[2], p[3]);
        if (t + 1 < SG_TERMS) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                x[2 * j] -= __uint_as_float(p[j] << 16);
                x[2 * j + 1] -= __uint_as_float(p[j] & 0xFFFF0000u);
            }
        }
    }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Operand chunk = rows [row0, row0 + 128) x contraction [k0, k0 + 16) of P: 256 pieces of 8 consecutive k of one row, one per
// converter thread.  The fp32 data travels global -> shared with cp.async into a slot only this thread reads back (a private
// FIFO: no barrier is involved and SG_FIFO - 1 chunks stay in flight per CTA without holding registers); out-of-range
// elements are zero-filled by the copy itself (src-size 0).
//   TR = false: P[(row0 + r) * ld + k], k contiguous: two 16-byte copies, slot = [half][thread] 16-byte words;
//   TR = true : P[k * ld + row0 + r], r contiguous: eight 4-byte copies (lanes over r: coalesced), slot = [j][thread] words.
template <bool TR>
__device__ __forceinline__ void sg_task(int t, int& r, int& kg) {
    if (!TR) { r = (t & 7) | ((t >> 4) << 3); kg = (t >> 3) & 1; }      // 8 lanes = 8 rows of one k group: conflict-free 16-byte stores
    else { r = t & 127; kg = t >> 7; }
}
template <bool TR>
__device__ __forceinline__ void sg_fetch(const float* __restrict__ P, int64_t ld, int64_t row0, int64_t rows, int64_t k0, int64_t kend,
                                         int tid, uint32_t slot_base) {
    int r, kg;
    sg_task<TR>(tid, r, kg);
    const int64_t row = row0 + r, k = k0 + kg * 8;
    if (!TR) {
        const bool ok = row < rows && k < kend;               // kend is a multiple of 8 on this path
        const float* src = ok ? P + row * ld + k : P;
        cp_async16(slot_base + tid * 16, src, ok ? 16u : 0u);
        cp_async16(slot_base + SG_CONV * 16 + tid * 16, src + 4, ok ? 16u : 0u);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool ok = row < rows && k + j < kend;
            cp_async4(slot_base + j * (SG_CONV * 4) + tid * 4, ok ? P + (k + j) * ld + row : P, ok ? 4u : 0u);
        }
    }
}
// read this thread's slot back, split, write the term images of the converted stage
template <bool TR, int ROWS = 128>       // ROWS: rows of the operand image this piece belongs to (k-group stride = 16 ROWS bytes)
__device__ __forceinline__ float sg_convert(const uint8_t* slot, uint8_t* img, int tid, int row_ofs = 0) {
    float x[8];
    if (!TR) {
        const float4 a = *reinterpret_cast<const float4*>(slot + tid * 16), b = *reinterpret_cast<const float4*>(slot + SG_CONV * 16 + tid * 16);
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = *reinterpret_cast<const float*>(slot + j * (SG_CONV * 4) + tid * 4);
    }
    const float sum8 = ((x[0] + x[1]) + (x[2] + x[3])) + ((x[4] + x[5]) + (x[6] + x[7]));      // wgrad: this piece of the bias gradient
    int r, kg;
    sg_task<TR>(tid, r, kg);
    uint4 terms[SG_TERMS];
    split8(x, terms);
#pragma unroll
    for (int t = 0; t < SG_TERMS; ++t) *reinterpret_cast<uint4*>(img + t * (ROWS * SG_BK * 2) + kg * (ROWS * 16) + (row_ofs + r) * 16) = terms[t];
    return sum8;
}

// BIMG: the B operand is a weight matrix whose term images were written once per optimiser step (split_pack_kernel): a
// producer thread bulk-copies the 4 KB term images of each chunk straight into the converted stage, and the converter
// threads only handle A.
template <bool AT, bool BT, int EPI, bool BIMG, int BN>
__global__ void __launch_bounds__(SG_THREADS, BN == 128 ? 2 : 1) split_gemm_kernel(const GemmArgs g, int tiles_n, int tiles_mn) {
    using Cfg = SgCfg<BN>;
    static_assert(BN == 128 || !BIMG, "weight images are tiled for 128 columns");
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar_empty = sbase + Cfg::kBarOfs;                               // per converted stage: its MMAs have completed
    const uint32_t bar_full = bar_empty + 8 * Cfg::kStages;                        // per converted stage: all pieces (and the weight image) written
    const uint32_t bar_done = bar_full + 8 * Cfg::kStages;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Cfg::kBarOfs + 64);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    int64_t tile = blockIdx.x;
    int64_t kbeg = 0, kend = g.Kdim;
    if (EPI == EPI_WGRAD) {
        const int64_t split = tile / tiles_mn;
        tile -= split * tiles_mn;
        kbeg = split * g.k_per_split;
        kend = kbeg + g.k_per_split < g.Kdim ? kbeg + g.k_per_split : g.Kdim;
    }
    const int64_t tn = tile % tiles_n;
    const int64_t m0 = (tile / tiles_n) * SG_BM, n0 = tn * BN;
    const int64_t nchunks = kend > kbeg ? (kend - kbeg + SG_BK - 1) / SG_BK : 0;

    // raw chunks 0 .. SG_FIFO-2 on their way before anything else
    auto fetch = [&](int64_t c) {
        if (c < nchunks && tid < SG_CONV) {
            const uint32_t slot = sbase + Cfg::kFifoOfs + (uint32_t)(c % SG_FIFO) * Cfg::kFifoSlot;
            sg_fetch<AT>(g.A, g.lda, m0, g.Mdim, kbeg + c * SG_BK, kend, tid, slot);
            if (!BIMG) {
#pragma unroll
                for (int h = 0; h < Cfg::kBTiles; ++h)
                    sg_fetch<BT>(g.B, g.ldb, n0 + 128 * h, g.Ndim, kbeg + c * SG_BK, kend, tid, slot + (1 + h) * SG_RAW_BYTES);
            }
        }
        cp_async_commit();                                   // one group per chunk index, possibly empty: keeps the wait count uniform
    };
#pragma unroll
    for (int c = 0; c < SG_FIFO - 1; ++c) fetch(c);

    if (tid == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(bar_empty + 8 * s, 1); mbar_init(bar_full + 8 * s, SG_CONV + (BIMG ? 1 : 0)); }
        mbar_init(bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == SG_CONV / 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(Cfg::kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // kind::f16, D = f32, A = B = bf16, both K-major, N = BN, M = 128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(SG_BM >> 4) << 24);
    const uint64_t dhi = desc_hi(2048, 128);          // LBO: between the two 8-wide k groups of the K = 16 step; SBO: between 8-row groups
    const uint64_t dhi_b = desc_hi(BN * 16, 128);     // the B image has BN rows per k group
    constexpr int kBTerm = BN * SG_BK * 2;            // bytes of one B term image
    if (tid < SG_CONV) {
        // ---- converters: raw FIFO -> bf16 term images of stage c % 2; nothing here waits for the MMA issue
        float colsum = 0.f;                                      // wgrad: sum over this CTA's points of dY[., m0 + r] (this thread's k group)
        for (int64_t c = 0; c < nchunks; ++c) {
            fetch(c + SG_FIFO - 1);                              // into the slot chunk c-1 was read from (same thread, program order)
            cp_async_wait<SG_FIFO - 1>();                        // chunk c has landed (this thread's copies are all this thread reads)
            const int s = (int)(c % Cfg::kStages);
            const int64_t use = c / Cfg::kStages;
            if (use > 0) mbar_wait(bar_empty + 8 * s, (uint32_t)((use - 1) & 1));      // the MMAs that read this stage have completed
            const uint8_t* slot = smem + Cfg::kFifoOfs + (c % SG_FIFO) * Cfg::kFifoSlot;
            uint8_t* stage = smem + s * Cfg::kStageBytes;
            colsum += sg_convert<AT>(slot, stage, tid);
            if (!BIMG) {
#pragma unroll
                for (int h = 0; h < Cfg::kBTiles; ++h)
                    sg_convert<BT, BN>(slot + (1 + h) * SG_RAW_BYTES, stage + SG_TERMS * SG_TERM_BYTES, tid, 128 * h);
            }
            fence_async_smem();
            mbar_arrive(bar_full + 8 * s);
        }
        // bias gradient = column sums of dY: the A pieces of a wgrad CTA are exactly that data; one column tile's CTAs report it
        if (EPI == EPI_WGRAD && g.colsum != nullptr && tn == 0 && nchunks > 0) {
            int r, kg;
            sg_task<AT>(tid, r, kg);
            if (m0 + r < g.Mdim) atomicAdd(g.colsum + m0 + r, colsum);
        }
    } else if (warp == SG_CONV / 32) {
        if (lane == 0) {
            // ---- MMA issuer
            for (int64_t c = 0; c < nchunks; ++c) {
                const int s = (int)(c % Cfg::kStages);
                mbar_wait(bar_full + 8 * s, (uint32_t)((c / Cfg::kStages) & 1));
                tc_fence_after();
                const uint32_t a0 = sbase + s * Cfg::kStageBytes, b0 = a0 + SG_TERMS * SG_TERM_BYTES;
                // Two accumulators.  tcgen05 adds each MMA into the fp32 accumulator with TRUNCATION (measured: same-sign sums
                // come out low by ~0.25 ulp per MMA, scripts/dbg_split_gemm.py), so the error grows with the number of MMAs that
                // touch an accumulator of full magnitude.  Only the x0 * y0 product (K / 16 MMAs) goes to the main accumulator;
                // the 5 cross products are 2^-8 .. 2^-16 of it and collect in their own accumulator,
                // where their truncation is that much smaller; the epilogue adds the two in registers (round to nearest).
#pragma unroll
                for (int sum = SG_TERMS - 1; sum >= 1; --sum) {          // smallest products first
#pragma unroll
                    for (int ta = 0; ta <= sum; ++ta) {
                        const int tb = sum - ta;
                        tc_mma(tmem_base + BN, desc_at(dhi, a0 + ta * SG_TERM_BYTES), desc_at(dhi_b, b0 + tb * kBTerm), idesc,
                               (c == 0 && sum == SG_TERMS - 1 && ta == 0) ? 0u : 1u);
                    }
                }
                tc_mma(tmem_base, desc_at(dhi, a0), desc_at(dhi_b, b0), idesc, c == 0 ? 0u : 1u);
                tc_commit(bar_empty + 8 * s);
                if (c + 1 == nchunks) tc_commit(bar_done);
            }
        }
    } else if (BIMG && lane == 0) {
        // ---- weight-image producer: chunk c of column tile tn = SG_TERMS contiguous 4 KB term images
        const uint8_t* img = g.b_img + ((size_t)tn * (size_t)(g.Kdim / SG_BK) + (size_t)(kbeg / SG_BK)) * SG_IMG_CHUNK;
        for (int64_t c = 0; c < nchunks; ++c) {
            const int s = (int)(c % Cfg::kStages);
            const int64_t use = c / Cfg::kStages;
            if (use > 0) mbar_wait(bar_empty + 8 * s, (uint32_t)((use - 1) & 1));
            mbar_expect_tx(bar_full + 8 * s, SG_IMG_CHUNK);
            bulk_g2s(sbase + s * Cfg::kStageBytes + SG_TERMS * SG_TERM_BYTES, img + (size_t)c * SG_IMG_CHUNK, SG_IMG_CHUNK, bar_full + 8 * s);
        }
    }
    cp_async_wait<0>();
    if (nchunks > 0 && tid < SG_CONV) {
        mbar_wait(bar_done, 0);
        tc_fence_after();
        // ---- epilogue, part 1: TMEM -> shared memory.  Thread = accumulator row (TMEM lane), warps 0-3 the first half of the
        // columns, warps 4-7 the second; main + cross added here.  The tile goes to the (now idle) stage / FIFO area as 128
        // rows of kEpiLd floats (padded: 16-byte stores of 8 consecutive rows hit 32 distinct banks).
        constexpr int LD = Cfg::kEpiLd;
        float* tile_s = reinterpret_cast<float*>(smem);
        {
            const int rowl = 32 * (warp & 3) + lane;
            const int cb = (BN / 2) * (warp >> 2);
#pragma unroll 1
            for (int cc = 0; cc < BN / 32; ++cc) {
                uint32_t v[16], vx[16];
                tc_ld16(tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(cb + 16 * cc), v);
                tc_ld16(tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(BN + cb + 16 * cc), vx);
                tc_wait_ld();
                pin16(v); pin16(vx);
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    *reinterpret_cast<float4*>(tile_s + rowl * LD + cb + 16 * cc + 4 * q) =
                        make_float4(__uint_as_float(v[4 * q]) + __uint_as_float(vx[4 * q]), __uint_as_float(v[4 * q + 1]) + __uint_as_float(vx[4 * q + 1]),
                                    __uint_as_float(v[4 * q + 2]) + __uint_as_float(vx[4 * q + 2]), __uint_as_float(v[4 * q + 3]) + __uint_as_float(vx[4 * q + 3]));
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(SG_CONV) : "memory");          // the 256 epilogue threads only
        // ---- part 2: shared memory -> global, one warp per row at a time, lane = 4 consecutive columns (512 contiguous bytes)
        const int64_t n = n0 + 4 * lane;
        if (EPI == EPI_WGRAD) {
            // split-K partial sums: one 128-byte run of atomics per instruction (lane = column)
            for (int r = warp; r < SG_BM; r += SG_CONV / 32) {
                const int64_t m = m0 + r;
                if (m >= g.Mdim) break;
#pragma unroll
                for (int q = 0; q < BN / 32; ++q) {
                    const int64_t nn = n0 + 32 * q + lane;
                    if (nn < g.n_valid) atomicAdd(g.C + m * g.ldc + nn, tile_s[r * LD + 32 * q + lane]);
                }
            }
        } else if (EPI == EPI_DGRAD && g.n_valid > 0) {
            // input gradients: columns < n_valid of an output with any row stride, one warp per row, lane = column
            for (int r = warp; r < SG_BM; r += SG_CONV / 32) {
                const int64_t m = m0 + r;
                if (m >= g.Mdim) break;
                for (int c = lane; c < BN; c += 32) {
                    const int64_t nn = n0 + c;
                    if (nn < g.n_valid) g.C[m * g.ldc + nn] = tile_s[r * LD + c] + (g.addend ? g.addend[m * g.ldadd + nn] : 0.f);
                }
            }
        } else if (BN == 128 && n < g.Ndim) {
            float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (EPI == EPI_FWD) bb = __ldg(reinterpret_cast<const float4*>(g.bias + n));
            for (int r = warp; r < SG_BM; r += SG_CONV / 32) {
                const int64_t m = m0 + r;
                if (m >= g.Mdim) break;
                float4 o = *reinterpret_cast<const float4*>(tile_s + r * LD + 4 * lane);
                if (EPI == EPI_FWD) {
                    o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
                    if (g.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                } else {
                    if (g.addend) {
                        const float4 ad = *reinterpret_cast<const float4*>(g.addend + m * g.ldadd + n);
                        o.x += ad.x; o.y += ad.y; o.z += ad.z; o.w += ad.w;
                    }
                    if (g.mask) {
                        const float4 mk = __ldg(reinterpret_cast<const float4*>(g.mask + m * g.ldm + n));
                        o.x = mk.x > 0.f ? o.x : 0.f; o.y = mk.y > 0.f ? o.y : 0.f;
                        o.z = mk.z > 0.f ? o.z : 0.f; o.w = mk.w > 0.f ? o.w : 0.f;
                    }
                }
                *reinterpret_cast<float4*>(g.C + m * g.ldc + n) = o;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == SG_CONV / 32) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
    }
}

// Term images of one weight matrix as the B operand of a role: B(n, k), n < n_rows (padded to 128-row tiles), k < k_len
// (a multiple of 16), element = W[n * ldw + k] (transpose = 0) or W[k * ldw + n] (transpose = 1), zero where k >= k_true
// (n >= n_true).  Layout: [n / 128][k / 16][term][(k / 8) % 2][n % 128][k % 8] bf16.
struct SplitPackJob { int64_t w_off; int ldw; int transpose; int n_true, k_true, n_tiles, k_chunks; size_t dst; };
constexpr int kSplitJobs = 22;
struct SplitPackArgs { SplitPackJob j[kSplitJobs]; };
__global__ void __launch_bounds__(256) split_pack_kernel(const float* __restrict__ params, uint8_t* __restrict__ base, const __grid_constant__ SplitPackArgs a) {
    const SplitPackJob& jb = a.j[blockIdx.y];
    const int64_t pieces = (int64_t)jb.n_tiles * jb.k_chunks * 256;              // (tile, chunk, k group, row)
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < pieces; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i & 127), kg = (int)((i >> 7) & 1);
        const int64_t tc_ = i >> 8;                                               // tile * k_chunks + chunk
        const int chunk = (int)(tc_ % jb.k_chunks), tile_n = (int)(tc_ / jb.k_chunks);
        const int n = tile_n * 128 + r, k0 = chunk * 16 + kg * 8;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = k0 + j;
            x[j] = (n < jb.n_true && k < jb.k_true) ? params[jb.w_off + (jb.transpose ? (int64_t)k * jb.ldw + n : (int64_t)n * jb.ldw + k)] : 0.f;
        }
        uint4 terms[SG_TERMS];
        split8(x, terms);
        uint8_t* dst = base + jb.dst + (size_t)tc_ * SG_IMG_CHUNK + kg * 2048 + r * 16;
#pragma unroll
        for (int t = 0; t < SG_TERMS; ++t) *reinterpret_cast<uint4*>(dst + t * SG_TERM_BYTES) = terms[t];
    }
}

template <bool AT, bool BT, int EPI, bool BIMG, int BN = 128>
static int launch_split_gemm(const GemmArgs& g, cudaStream_t st) {
    using Cfg = SgCfg<BN>;
    auto kern = split_gemm_kernel<AT, BT, EPI, BIMG, BN>;
    static bool configured = false;          // per instantiation
    if (!configured) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(split_gemm_kernel)");
        configured = true;
    }
    const int64_t tiles_m = cdiv(g.Mdim, SG_BM), tiles_n = cdiv(g.Ndim, BN);
    int64_t splits = 1;
    GemmArgs a = g;
    if (EPI == EPI_WGRAD) {
        // split the contraction (points) so that every SM holds its two CTAs (one for BN = 256); k_per_split a multiple of the chunk
        int64_t want = (int64_t)num_sms() * (BN == 128 ? 2 : 1) / (tiles_m * tiles_n);
        if (want < 1) want = 1;
        int64_t kps = cdiv(cdiv(g.Kdim, want), SG_BK) * SG_BK;
        if (kps < 256) kps = 256;
        splits = cdiv(g.Kdim, kps);
        a.k_per_split = kps;
    }
    const int64_t grid = tiles_m * tiles_n * splits;
    if (grid <= 0) return NSB_OK;
    if (grid > 0x7fffffffLL) return NSB_E_BADARG;
    kern<<<(unsigned)grid, SG_THREADS, Cfg::kSmemBytes, st>>>(a, (int)tiles_n, (int)(tiles_m * tiles_n));
    NSB_LAUNCH_CHECK("split_gemm_kernel");
    return NSB_OK;
}

}  // namespace tc

size_t split_image_bytes(int n_rows, int k_len) { return (size_t)cdiv(n_rows, 128) * (size_t)(k_len / 16) * tc::SG_IMG_CHUNK; }

// Every weight image of a net: forward B = W (n = out feature, k = in feature, zero beyond K), dgrad B = W^T restricted to
// the first 256 in features (n = in feature, k = out feature), and W^T of the three input slices.  One launch, 22 jobs; ~7 MB
// written per net.
int split_pack(const float* params, void* packed, cudaStream_t st) {
    const PackedLayout L = packed_layout();
    tc::SplitPackArgs a;
    int nj = 0;
    for (int l = 0; l < 12; ++l) {
        if (l == 9 || l == 11) continue;
        const LayerDesc d = layer_desc(l);
        a.j[nj++] = tc::SplitPackJob{d.w_off, d.K, 0, d.N, d.K, (int)cdiv(d.N, 128), d.Kpad / 16, L.split_fwd[l]};
        if (l > 0) a.j[nj++] = tc::SplitPackJob{d.w_off, d.K, 1, kHidden, d.N, kHidden / 128, d.N / 16, L.split_dgrad[l]};
    }
    // input slices (dgrad B = W^T rows n = in feature): gamma(x) columns of mlp.0 and mlp.4, gamma(d) columns of color_fc
    const LayerDesc d0 = layer_desc(0), d4 = layer_desc(4), dc = layer_desc(10);
    a.j[nj++] = tc::SplitPackJob{d0.w_off, d0.K, 1, kPosDim, d0.N, 1, d0.N / 16, L.split_dinput[0]};
    a.j[nj++] = tc::SplitPackJob{d4.w_off + kHidden, d4.K, 1, kPosDim, d4.N, 1, d4.N / 16, L.split_dinput[1]};
    a.j[nj++] = tc::SplitPackJob{dc.w_off + kHidden, dc.K, 1, kDirDim, dc.N, 1, dc.N / 16, L.split_dinput[2]};
    if (nj != tc::kSplitJobs) return NSB_E_BADARG;
    tc::split_pack_kernel<<<dim3(16, tc::kSplitJobs), 256, 0, st>>>(params, reinterpret_cast<uint8_t*>(packed), a);
    NSB_LAUNCH_CHECK("split_pack_kernel");
    return NSB_OK;
}

int split_gemm(const GemmArgs& g, int role, cudaStream_t st) {
    NSB_TRY(check_arch());
    // alignment contract of the loaders / epilogues (all layer buffers of field_fp32.cu satisfy it)
    const bool any_ldc = role == EPI_DGRAD && g.n_valid > 0;        // input gradients: scalar epilogue, any row stride
    if ((g.lda & 3) || (g.ldb & 3) || (role != EPI_WGRAD && ((g.Kdim & 15) || ((g.ldc & 3) && !any_ldc) || (g.Ndim & 15)))) return NSB_E_BADARG;
    const bool img = g.b_img != nullptr && role != EPI_WGRAD;
    switch (role) {
        case EPI_FWD: return img ? tc::launch_split_gemm<false, false, EPI_FWD, true>(g, st) : tc::launch_split_gemm<false, false, EPI_FWD, false>(g, st);
        case EPI_DGRAD: return img ? tc::launch_split_gemm<false, true, EPI_DGRAD, true>(g, st) : tc::launch_split_gemm<false, true, EPI_DGRAD, false>(g, st);
        case EPI_WGRAD: {
            // 256-column CTAs over the whole multiples of 256 columns of B, 128-column CTAs over the rest (gamma(x) / gamma(d)
            // columns of the skip and colour layers, layer 0); the bias gradient rides with the first launch only
            const int64_t wide = g.Ndim / 256 * 256;
            if (wide > 0) {
                GemmArgs a = g;
                a.Ndim = wide; a.n_valid = g.n_valid < wide ? g.n_valid : (int)wide;
                NSB_TRY((tc::launch_split_gemm<true, true, EPI_WGRAD, false, 256>(a, st)));
            }
            if (wide < g.Ndim) {
                GemmArgs a = g;
                a.B = g.B + wide; a.C = g.C + wide; a.Ndim = g.Ndim - wide; a.n_valid = g.n_valid - (int)wide;
                if (wide > 0) a.colsum = nullptr;
                if (a.n_valid > 0) return tc::launch_split_gemm<true, true, EPI_WGRAD, false, 128>(a, st);
            }
            return NSB_OK;
        }
    }
    return NSB_E_BADARG;
}

}  // namespace nsb

// Test hook (not in include/nsb.h): one GEMM of the given role on caller buffers.
extern "C" int nsb_debug_split_gemm(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                                    int64_t N, int64_t K, int role, const float* bias, int relu, const float* mask, int64_t ldm,
                                    const float* addend, int64_t ldadd, int n_valid, float* colsum, void* stream) {
    nsb::GemmArgs g{};
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc; g.Mdim = M; g.Ndim = N; g.Kdim = K;
    g.bias = bias; g.relu = relu; g.mask = mask; g.ldm = ldm; g.addend = addend; g.ldadd = ldadd; g.n_valid = n_valid; g.colsum = colsum;
    return nsb::split_gemm(g, role, nsb::as_stream(stream));
}
