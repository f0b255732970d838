// gemv_mma.cu -- skinny path, 3 <= T <= 8 tokens per pass: the decode weight stream of gemv.cu
// with the integer dots on the legacy tensor path (mma.sync.m16n8k32, s32 += u8 x s8, IMMA.16832).
//
// Why: the dp4a GEMV spends ~20 instructions per block per TOKEN and turns compute-bound from
// T = 3 (SURVEY.md section 7, hard part 4).  One m16n8k32 does 16 weight rows x 8 tokens x one
// quantization block; tokens sit on the 8-wide N side, so T = 3..8 costs the same as T = 1.
// K = 32 per instruction = one block, so the s32 fragment IS sumi[16 rows][8 tokens] of that block
// and the reference's per-block fold (qgemm_common.cuh) is applied to it in registers.
//
//   * two CTAs per SM; producer warp streams tiles of 16 weight rows (one bulk copy per row into a
//     padded smem pitch, so the 8 row-groups of a fragment load hit different banks)
//   * 8 consumer warps split K: warp w owns blocks [w*NBW, (w+1)*NBW) of all 16 rows, its
//     activation fragments (2 registers per block) live in registers for the whole kernel
//   * per tile: 8 partial 16x8 tiles are combined through smem in warp order (deterministic)
#include "ptx.cuh"
#include "qgemm_common.cuh"

namespace qgemm {

constexpr int kMmaWarps = 8;
constexpr int kMmaThreads = (kMmaWarps + 1) * 32;
constexpr int kMmaRows = 16;          // weight rows per tile = MMA M
constexpr int kMmaStagesMax = 6;
constexpr int kMmaSmemBudget = 112 * 1024;   // two CTAs per SM when two stages fit in this
constexpr int kMmaSmemMax = 200 * 1024;      // otherwise one CTA per SM (long or 8-bit rows)

struct GemvMmaParams {
    const uint8_t* act;
    const uint8_t* wgt;
    float* C;
    int T, F, nb;
    int64_t ldc_t, ldc_f;
    int pitch;        // smem bytes per row segment of one chunk (+ 16: pitch % 128 == 16)
    int stages;
    int pdl;
    int span;         // tuning aid: split rows, not tiles, over the CTAs
    PeerOut peer;
};

__device__ __forceinline__ void mma_u8s8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_s8s8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// A-fragment registers of one weight row for thread-in-group `tig`:
//   lo = elements 4*tig .. 4*tig+3, hi = elements 16+4*tig .. 16+4*tig+3   (un-offset u8, or s8 for q8_0)
//   al4: the block's quant words are 4-byte aligned in smem (known at compile time after unrolling: one word load
//   instead of two halves)
__device__ __forceinline__ uint32_t ld_u32_sel(const uint8_t* p, bool al4) {
    return al4 ? *reinterpret_cast<const uint32_t*>(p) : ld_u32_a2(p);
}
template <int WT>
__device__ __forceinline__ void row_frag(const uint8_t* blk, int tig, uint32_t& lo, uint32_t& hi, WScale& ws,
                                         bool al4 = false) {
    using Fm = Fmt<WT>;
    ws = load_wscale<WT>(blk);
    if constexpr (Fm::bits == 8) {
        lo = ld_u32_sel(blk + Fm::qs + 4 * tig, al4);
        hi = ld_u32_sel(blk + Fm::qs + 16 + 4 * tig, al4);
    } else {
        const uint32_t v = ld_u32_sel(blk + Fm::qs + 4 * tig, al4);
        lo = v & 0x0f0f0f0fu;
        hi = (v >> 4) & 0x0f0f0f0fu;
        if constexpr (Fm::bits == 5) {
            const uint32_t qh = ld_u32_sel(blk + Fm::qh, al4);
            lo |= spread_qh4(qh, 4 * tig);
            hi |= spread_qh4(qh, 16 + 4 * tig);
        }
    }
}

// K-chunks per row for a given format and register-fragment depth: the smallest split that leaves room for
// four stages with two CTAs per SM (whole-row stages of the 8-bit and 5-bit formats did not, which cost them
// half the resident warps)
constexpr int mma_pitch(int seg) { return seg + 16 + ((128 - (seg % 128)) % 128); }
constexpr size_t mma_fixed(int nb) { return 128 + kMmaWarps * 128 * 4 + (size_t)nb * 64 + 128; }
constexpr int mma_pick_nc(int bytes, int nbw) {
    // whole rows when two stages of them fit (measured: chunking costs the 4-bit formats ~5 %)
    if (mma_fixed(nbw * kMmaWarps) + 2 * (size_t)kMmaRows * mma_pitch(nbw * kMmaWarps * bytes) <= (size_t)kMmaSmemBudget) return 1;
    for (int nc = 2; nc <= 8; nc *= 2) {
        if (nbw % nc) break;
        const int seg = (nbw / nc) * kMmaWarps * bytes;
        if (mma_fixed(nbw * kMmaWarps) + 4 * (size_t)kMmaRows * mma_pitch(seg) <= (size_t)kMmaSmemBudget) return nc;
    }
    return nbw >= 8 ? 8 : nbw;
}

// NBW = K-blocks per warp held as register fragments, NC = K-chunks a row is streamed in.
// A CTA owns a contiguous span of weight rows at one-row granularity (so every CTA streams the same number
// of bytes), walked in tiles of up to 16 rows; chunk c of a tile holds blocks [c*CB, (c+1)*CB) of each row and
// warp w owns blocks c*CB + w*PER .. + PER-1 of every chunk.
// kFull: nb == 8 * NBW, every (chunk, block) slot is real -- no guards in the unrolled loops, so the loads of
// the next block move above the MMA of this one.
template <int WT, int NBW, int NC, bool kMsExact, bool kFull>
__global__ void __launch_bounds__(kMmaThreads, 2) gemv_mma_kernel(const GemvMmaParams p) {
    using Fm = Fmt<WT>;
    constexpr int PER = NBW / NC;
    constexpr int CB = PER * kMmaWarps;
    // quant words of block i of a warp's slice are word-aligned when the slice starts word-aligned and ...
    constexpr bool kSliceAl = (PER * Fm::bytes) % 4 == 0;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int nb = p.nb;

    uint64_t* full = reinterpret_cast<uint64_t*>(smem);         // [kMmaStagesMax]
    uint64_t* empty = full + kMmaStagesMax;                     // [kMmaStagesMax]
    float* red = reinterpret_cast<float*>(smem + 128);          // [kMmaWarps][16 rows][8 tokens]
    float2* a_sc = reinterpret_cast<float2*>(smem + 128 + kMmaWarps * 128 * 4);  // [nb][8] (d_a, c_a)
    const uint32_t stage_bytes = (uint32_t)kMmaRows * p.pitch;
    uint8_t* stage0 = smem + ((128u + kMmaWarps * 128u * 4u + (uint32_t)nb * 64u + 127u) & ~127u);

    // whole 16-row tiles per CTA: the kernel is issue-bound, so no CTA should spend MMAs on rows it does not own
    // (p.span: one-row granularity instead -- equal bytes per CTA, more MMAs; tuning aid)
    const int ntiles_total = (p.F + kMmaRows - 1) / kMmaRows;
    const int r_begin = p.span ? (int)(((int64_t)p.F * blockIdx.x) / gridDim.x)
                               : kMmaRows * (int)(((int64_t)ntiles_total * blockIdx.x) / gridDim.x);
    const int r_end = p.span ? (int)(((int64_t)p.F * (blockIdx.x + 1)) / gridDim.x)
                             : min(p.F, kMmaRows * (int)(((int64_t)ntiles_total * (blockIdx.x + 1)) / gridDim.x));
    const size_t rowbytes = (size_t)nb * Fm::bytes;

    if (tid == 0) {
        for (int s = 0; s < p.stages; s++) {
            ptx::mbar_init(&full[s], 1);
            ptx::mbar_init(&empty[s], kMmaWarps);
        }
        ptx::fence_mbar_init();
    }
    __syncthreads();
    if (p.pdl) ptx::griddep_launch_dependents();

    if (warp == kMmaWarps) {
        // ===== producer: per chunk, one bulk copy per weight row of the tile into the padded pitch
        int s = 0;
        uint32_t ph = 0;
        for (int r = r_begin; r < r_end; r += kMmaRows) {
            const int nrows = min(kMmaRows, r_end - r);   // rows beyond keep stale smem: computed, never stored
            for (int c = 0; c < NC; c++) {
                const int cb = min(CB, nb - c * CB);
                if (cb <= 0) break;
                const uint32_t seg = (uint32_t)cb * Fm::bytes;
                ptx::mbar_wait(&empty[s], ph ^ 1);
                if (lane == 0) ptx::mbar_arrive_expect_tx(&full[s], seg * (uint32_t)nrows);
                __syncwarp();
                if (lane < nrows)
                    ptx::bulk_g2s(stage0 + (size_t)s * stage_bytes + (size_t)lane * p.pitch,
                                  p.wgt + (size_t)(r + lane) * rowbytes + (size_t)c * CB * Fm::bytes, seg, &full[s]);
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
        }
        return;
    }

    // ===== consumers
    if (p.pdl == 1) ptx::griddep_wait();
    if (p.peer.world > 1) {
        if (tid == 0) peer_wait_prior(p.peer);
        ptx::bar_sync(1, kMmaWarps * 32);
    }
    // B fragments: token g (zero beyond T), elements 4*tig.. and 16+4*tig.. of each of this warp's blocks
    uint32_t bf[NBW][2];
#pragma unroll
    for (int c = 0; c < NC; c++) {
#pragma unroll
        for (int i = 0; i < PER; i++) {
            const int b = c * CB + warp * PER + i;
            bf[c * PER + i][0] = bf[c * PER + i][1] = 0u;
            if ((kFull || b < nb) && g < p.T) {
                const uint32_t* q = reinterpret_cast<const uint32_t*>(p.act + ((size_t)g * nb + b) * kQ81Bytes);
                bf[c * PER + i][0] = __ldg(q + 1 + tig);
                bf[c * PER + i][1] = __ldg(q + 5 + tig);
            }
        }
    }
    // activation scales of all blocks, all 8 token slots: [b][token] (d_a, c_a)
    for (int i = tid; i < nb * 8; i += kMmaWarps * 32) {
        const int b = i >> 3, t = i & 7;
        ActScale sc{0.f, 0.f};
        if (t < p.T) {
            const uint32_t ds = __ldg(reinterpret_cast<const uint32_t*>(p.act + ((size_t)t * nb + b) * kQ81Bytes));
            sc = prep_act_scale<WT, kMsExact>(half_bits_to_float(ds), half_bits_to_float(ds >> 16));
        }
        a_sc[i] = make_float2(sc.d, sc.s);
    }
    ptx::bar_sync(1, kMmaWarps * 32);

    int s = 0;
    uint32_t ph = 0;
    for (int r = r_begin; r < r_end; r += kMmaRows) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};  // (row g, tok 2tig), (row g, tok 2tig+1), (row g+8, ...)
#pragma unroll
        for (int c = 0; c < NC; c++) {
            if (kFull || c * CB < nb) {
                ptx::mbar_wait(&full[s], ph);
                const uint8_t* r0 = stage0 + (size_t)s * stage_bytes + (size_t)g * p.pitch + (size_t)(warp * PER) * Fm::bytes;
                const uint8_t* r1 = r0 + (size_t)8 * p.pitch;
#pragma unroll
                for (int i = 0; i < PER; i++) {
                    const int b = c * CB + warp * PER + i;
                    if (kFull || b < nb) {
                        uint32_t a[4];
                        WScale w0, w1;
                        // ... the block's own offset keeps the quant words on a word boundary
                        const bool al4 = kSliceAl && (i * Fm::bytes + Fm::qs) % 4 == 0 &&
                                         (Fm::bits != 5 || (i * Fm::bytes + Fm::qh) % 4 == 0);
                        row_frag<WT>(r0 + (size_t)i * Fm::bytes, tig, a[0], a[2], w0, al4);
                        row_frag<WT>(r1 + (size_t)i * Fm::bytes, tig, a[1], a[3], w1, al4);
                        int cc[4] = {0, 0, 0, 0};
                        if constexpr (Fm::bits == 8) mma_s8s8(cc, a, bf[c * PER + i][0], bf[c * PER + i][1]);
                        else mma_u8s8(cc, a, bf[c * PER + i][0], bf[c * PER + i][1]);
                        const float4 sc = *reinterpret_cast<const float4*>(&a_sc[b * 8 + 2 * tig]);  // tokens 2tig, 2tig+1
                        acc[0] = fold_block_pre<WT>(acc[0], cc[0], w0, ActScale{sc.x, sc.y});
                        acc[1] = fold_block_pre<WT>(acc[1], cc[1], w0, ActScale{sc.z, sc.w});
                        acc[2] = fold_block_pre<WT>(acc[2], cc[2], w1, ActScale{sc.x, sc.y});
                        acc[3] = fold_block_pre<WT>(acc[3], cc[3], w1, ActScale{sc.z, sc.w});
                    }
                }
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&empty[s]);
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
        }

        // combine the 8 K-slices in warp order
        float* rb = red;
        rb[warp * 128 + g * 8 + 2 * tig] = acc[0];
        rb[warp * 128 + g * 8 + 2 * tig + 1] = acc[1];
        rb[warp * 128 + (g + 8) * 8 + 2 * tig] = acc[2];
        rb[warp * 128 + (g + 8) * 8 + 2 * tig + 1] = acc[3];
        ptx::bar_sync(1, kMmaWarps * 32);
        if (tid < 128) {
            const int row = tid >> 3, tok = tid & 7;
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kMmaWarps; w++) v += rb[w * 128 + tid];
            const int f = r + row;
            if (f < r_end && tok < p.T) peer_store(p.peer, p.C, (int64_t)tok * p.ldc_t + (int64_t)f * p.ldc_f, v);
        }
        ptx::bar_sync(1, kMmaWarps * 32);  // the partials buffer is reused by the next tile
    }
    if (p.peer.world > 1) {
        if (!(p.peer.dbg & 4)) __threadfence();  // this thread's peer stores are ordered before the CTA barrier
        ptx::bar_sync(1, kMmaWarps * 32);
        if (tid == 0) peer_signal_done(p.peer, gridDim.x);
    }
    if (p.pdl == 2) ptx::griddep_wait();
}

// ---------------------------------------------------------------------------
// Long rows (K > 8192): the same mapping with the activation fragments in shared memory and
// the 16-row tile streamed in K-chunks, so neither registers nor one stage have to hold a row.
//   smem: [barriers | partials | a_sc[nb][8] | frag[nb][32 lanes] (2 words) | stages of 16 x chunk]
// ---------------------------------------------------------------------------
constexpr int kBigChunk = 64;   // K-blocks per stage (multiple of 8: row segments stay 16-byte multiples)

struct GemvMmaBigParams {
    const uint8_t* act;
    const uint8_t* wgt;
    float* C;
    int T, F, nb;
    int64_t ldc_t, ldc_f;
    int pitch;        // smem bytes per row segment (kBigChunk blocks + pad, pitch % 128 == 16)
    int stages;
    int pdl;
    PeerOut peer;
};

template <int WT, bool kMsExact>
__global__ void __launch_bounds__(kMmaThreads, 1) gemv_mma_bigk_kernel(const GemvMmaBigParams p) {
    using Fm = Fmt<WT>;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int nb = p.nb;

    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty = full + kMmaStagesMax;
    float* red = reinterpret_cast<float*>(smem + 128);                                   // [kMmaWarps][128]
    float2* a_sc = reinterpret_cast<float2*>(smem + 128 + kMmaWarps * 128 * 4);          // [nb][8]
    uint2* frag = reinterpret_cast<uint2*>(smem + 128 + kMmaWarps * 128 * 4 + (size_t)nb * 64);  // [nb][32]
    const uint32_t stage_bytes = (uint32_t)kMmaRows * p.pitch;
    uint8_t* stage0 = smem + ((128u + kMmaWarps * 128u * 4u + (uint32_t)nb * 320u + 127u) & ~127u);

    const int ntiles_total = (p.F + kMmaRows - 1) / kMmaRows;
    const int t_begin = (int)(((int64_t)ntiles_total * blockIdx.x) / gridDim.x);
    const int t_end = (int)(((int64_t)ntiles_total * (blockIdx.x + 1)) / gridDim.x);
    const size_t rowbytes = (size_t)nb * Fm::bytes;
    const int nchunks = (nb + kBigChunk - 1) / kBigChunk;

    if (tid == 0) {
        for (int s = 0; s < p.stages; s++) {
            ptx::mbar_init(&full[s], 1);
            ptx::mbar_init(&empty[s], kMmaWarps);
        }
        ptx::fence_mbar_init();
    }
    __syncthreads();
    if (p.pdl) ptx::griddep_launch_dependents();

    if (warp == kMmaWarps) {
        int s = 0;
        uint32_t ph = 0;
        for (int t = t_begin; t < t_end; t++) {
            for (int c = 0; c < nchunks; c++) {
                const int cb = min(kBigChunk, nb - c * kBigChunk);
                const uint32_t seg = (uint32_t)cb * Fm::bytes;
                ptx::mbar_wait(&empty[s], ph ^ 1);
                if (lane == 0) ptx::mbar_arrive_expect_tx(&full[s], seg * kMmaRows);
                __syncwarp();
                if (lane < kMmaRows) {
                    const int f = min(t * kMmaRows + lane, p.F - 1);
                    ptx::bulk_g2s(stage0 + (size_t)s * stage_bytes + (size_t)lane * p.pitch,
                                  p.wgt + (size_t)f * rowbytes + (size_t)c * kBigChunk * Fm::bytes, seg, &full[s]);
                }
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
        }
        return;
    }

    if (p.pdl == 1) ptx::griddep_wait();
    if (p.peer.world > 1) {
        if (tid == 0) peer_wait_prior(p.peer);
        ptx::bar_sync(1, kMmaWarps * 32);
    }
    for (int b = warp; b < nb; b += kMmaWarps) {   // fragments of token g: elements 4*tig.. and 16+4*tig..
        uint2 v = make_uint2(0u, 0u);
        if (g < p.T) {
            const uint32_t* q = reinterpret_cast<const uint32_t*>(p.act + ((size_t)g * nb + b) * kQ81Bytes);
            v.x = __ldg(q + 1 + tig);
            v.y = __ldg(q + 5 + tig);
        }
        frag[b * 32 + lane] = v;
    }
    for (int i = tid; i < nb * 8; i += kMmaWarps * 32) {
        const int b = i >> 3, t = i & 7;
        ActScale sc{0.f, 0.f};
        if (t < p.T) {
            const uint32_t ds = __ldg(reinterpret_cast<const uint32_t*>(p.act + ((size_t)t * nb + b) * kQ81Bytes));
            sc = prep_act_scale<WT, kMsExact>(half_bits_to_float(ds), half_bits_to_float(ds >> 16));
        }
        a_sc[i] = make_float2(sc.d, sc.s);
    }
    ptx::bar_sync(1, kMmaWarps * 32);

    int s = 0;
    uint32_t ph = 0;
    for (int t = t_begin; t < t_end; t++) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < nchunks; c++) {
            const int cb = min(kBigChunk, nb - c * kBigChunk);
            ptx::mbar_wait(&full[s], ph);
            const uint8_t* r0 = stage0 + (size_t)s * stage_bytes + (size_t)g * p.pitch;
            const uint8_t* r1 = r0 + (size_t)8 * p.pitch;
#pragma unroll 2
            for (int i = warp; i < cb; i += kMmaWarps) {
                const int b = c * kBigChunk + i;
                uint32_t a[4];
                WScale w0, w1;
                row_frag<WT>(r0 + (size_t)i * Fm::bytes, tig, a[0], a[2], w0);
                row_frag<WT>(r1 + (size_t)i * Fm::bytes, tig, a[1], a[3], w1);
                const uint2 bfr = frag[b * 32 + lane];
                int cc[4] = {0, 0, 0, 0};
                if constexpr (Fm::bits == 8) mma_s8s8(cc, a, bfr.x, bfr.y);
                else mma_u8s8(cc, a, bfr.x, bfr.y);
                const float4 sc = *reinterpret_cast<const float4*>(&a_sc[b * 8 + 2 * tig]);
                acc[0] = fold_block_pre<WT>(acc[0], cc[0], w0, ActScale{sc.x, sc.y});
                acc[1] = fold_block_pre<WT>(acc[1], cc[1], w0, ActScale{sc.z, sc.w});
                acc[2] = fold_block_pre<WT>(acc[2], cc[2], w1, ActScale{sc.x, sc.y});
                acc[3] = fold_block_pre<WT>(acc[3], cc[3], w1, ActScale{sc.z, sc.w});
            }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&empty[s]);
            if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        red[warp * 128 + g * 8 + 2 * tig] = acc[0];
        red[warp * 128 + g * 8 + 2 * tig + 1] = acc[1];
        red[warp * 128 + (g + 8) * 8 + 2 * tig] = acc[2];
        red[warp * 128 + (g + 8) * 8 + 2 * tig + 1] = acc[3];
        ptx::bar_sync(1, kMmaWarps * 32);
        if (tid < 128) {
            const int r = tid >> 3, tok = tid & 7;
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kMmaWarps; w++) v += red[w * 128 + tid];
            const int f = t * kMmaRows + r;
            if (f < p.F && tok < p.T) peer_store(p.peer, p.C, (int64_t)tok * p.ldc_t + (int64_t)f * p.ldc_f, v);
        }
        ptx::bar_sync(1, kMmaWarps * 32);
    }
    if (p.peer.world > 1) {
        if (!(p.peer.dbg & 4)) __threadfence();
        ptx::bar_sync(1, kMmaWarps * 32);
        if (tid == 0) peer_signal_done(p.peer, gridDim.x);
    }
    if (p.pdl == 2) ptx::griddep_wait();
}

// ---------------------------------------------------------------------------
// Small batches, 9 <= T (passes of 8*NT tokens): the same weight stream with NT token tiles per pass, so a
// weight fragment is unpacked once and feeds NT MMAs.  One CTA per SM, 16 consumer warps splitting K (NBW blocks
// each, nb == 16 * NBW exactly), B fragments of all NT tiles in registers (NBW * NT * 2), whole 16-row tiles per
// stage.  The CTA-wide barrier that ends a tile's reduction also proves its stage free, so thread 0 refills it right
// there and no producer warp or "empty" barriers are needed.  Passes of 8 through the kernel above re-stream (from L2) and re-unpack the weights for every 8 tokens:
// q4_0 11008x4096 T=32 took 36 us that way.
// ---------------------------------------------------------------------------
constexpr int kWideWarps = 16;
constexpr int kWideThreads = kWideWarps * 32;   // no producer warp: 4 warps per SM sub-partition leave 128 registers per thread
constexpr int kWideRedPitch = 40;   // floats per row of a warp's partial tile (32 tokens + pad: 2-way conflicts at most)
constexpr int kWideSmemMax = 220 * 1024;

struct GemvMmaWideParams {
    const uint8_t* act;
    const uint8_t* wgt;
    float* C;
    int T, F, nb;         // T <= 8 * NT tokens of this pass
    int64_t ldc_t, ldc_f;
    int pitch, stages, pdl;
};

template <int WT, int NBW, int NT, bool kMsExact>
__global__ void __launch_bounds__(kWideThreads, 1) gemv_mma_wide_kernel(const GemvMmaWideParams p) {
    using Fm = Fmt<WT>;
    constexpr int TOK = 8 * NT;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int nb = p.nb;

    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    float* red = reinterpret_cast<float*>(smem + 128);                                    // [16 warps][16 rows][kWideRedPitch]
    constexpr uint32_t kRedBytes = kWideWarps * kMmaRows * kWideRedPitch * 4;
    float2* a_sc = reinterpret_cast<float2*>(smem + 128 + kRedBytes);                     // [nb][TOK] (d_a, c_a)
    const uint32_t stage_bytes = (uint32_t)kMmaRows * p.pitch;
    uint8_t* stage0 = smem + ((128u + kRedBytes + (uint32_t)nb * TOK * 8u + 127u) & ~127u);

    const int ntiles_total = (p.F + kMmaRows - 1) / kMmaRows;
    const int t_begin = (int)(((int64_t)ntiles_total * blockIdx.x) / gridDim.x);
    const int t_end = (int)(((int64_t)ntiles_total * (blockIdx.x + 1)) / gridDim.x);
    const size_t rowbytes = (size_t)nb * Fm::bytes;

    // one thread streams: tile `t` of this CTA goes to stage (t - t_begin) % stages, one bulk copy per weight row
    auto issue_tile = [&](int t) {
        const int st = (t - t_begin) % p.stages;
        ptx::mbar_arrive_expect_tx(&full[st], (uint32_t)(kMmaRows * rowbytes));
        for (int r = 0; r < kMmaRows; r++) {
            const int f = min(t * kMmaRows + r, p.F - 1);  // tail tile: re-read a valid row, never stored
            ptx::bulk_g2s(stage0 + (size_t)st * stage_bytes + (size_t)r * p.pitch, p.wgt + (size_t)f * rowbytes,
                          (uint32_t)rowbytes, &full[st]);
        }
    };
    if (tid == 0) {
        for (int s = 0; s < p.stages; s++) ptx::mbar_init(&full[s], 1);
        ptx::fence_mbar_init();
        for (int t = t_begin; t < min(t_end, t_begin + p.stages); t++) issue_tile(t);   // weights never depend on the predecessor
    }
    __syncthreads();
    if (p.pdl) ptx::griddep_launch_dependents();

    if (p.pdl == 1) ptx::griddep_wait();
    // B fragments: token 8j + g of tile j (zero beyond T), this warp's NBW blocks
    uint32_t bf[NBW][NT][2];
#pragma unroll
    for (int i = 0; i < NBW; i++) {
        const int b = warp * NBW + i;
#pragma unroll
        for (int j = 0; j < NT; j++) {
            const int tok = 8 * j + g;
            bf[i][j][0] = bf[i][j][1] = 0u;
            if (tok < p.T) {
                const uint32_t* q = reinterpret_cast<const uint32_t*>(p.act + ((size_t)tok * nb + b) * kQ81Bytes);
                bf[i][j][0] = __ldg(q + 1 + tig);
                bf[i][j][1] = __ldg(q + 5 + tig);
            }
        }
    }
    for (int i = tid; i < nb * TOK; i += kWideWarps * 32) {
        const int b = i / TOK, t = i - b * TOK;
        ActScale sc{0.f, 0.f};
        if (t < p.T) {
            const uint32_t ds = __ldg(reinterpret_cast<const uint32_t*>(p.act + ((size_t)t * nb + b) * kQ81Bytes));
            sc = prep_act_scale<WT, kMsExact>(half_bits_to_float(ds), half_bits_to_float(ds >> 16));
        }
        a_sc[i] = make_float2(sc.d, sc.s);
    }
    ptx::bar_sync(1, kWideWarps * 32);

    constexpr bool kSliceAl = (NBW * Fm::bytes) % 4 == 0;
    int s = 0;
    uint32_t ph = 0;
    for (int t = t_begin; t < t_end; t++) {
        ptx::mbar_wait(&full[s], ph);
        const uint8_t* r0 = stage0 + (size_t)s * stage_bytes + (size_t)g * p.pitch + (size_t)(warp * NBW) * Fm::bytes;
        const uint8_t* r1 = r0 + (size_t)8 * p.pitch;
        float acc[NT][4];
#pragma unroll
        for (int j = 0; j < NT; j++) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
#pragma unroll
        for (int i = 0; i < NBW; i++) {
            const int b = warp * NBW + i;
            uint32_t a[4];
            WScale w0, w1;
            const bool al4 = kSliceAl && (i * Fm::bytes + Fm::qs) % 4 == 0 && (Fm::bits != 5 || (i * Fm::bytes + Fm::qh) % 4 == 0);
            row_frag<WT>(r0 + (size_t)i * Fm::bytes, tig, a[0], a[2], w0, al4);
            row_frag<WT>(r1 + (size_t)i * Fm::bytes, tig, a[1], a[3], w1, al4);
#pragma unroll
            for (int j = 0; j < NT; j++) {
                int cc[4] = {0, 0, 0, 0};
                if constexpr (Fm::bits == 8) mma_s8s8(cc, a, bf[i][j][0], bf[i][j][1]);
                else mma_u8s8(cc, a, bf[i][j][0], bf[i][j][1]);
                const float4 sc = *reinterpret_cast<const float4*>(&a_sc[b * TOK + 8 * j + 2 * tig]);
                acc[j][0] = fold_block_pre<WT>(acc[j][0], cc[0], w0, ActScale{sc.x, sc.y});
                acc[j][1] = fold_block_pre<WT>(acc[j][1], cc[1], w0, ActScale{sc.z, sc.w});
                acc[j][2] = fold_block_pre<WT>(acc[j][2], cc[2], w1, ActScale{sc.x, sc.y});
                acc[j][3] = fold_block_pre<WT>(acc[j][3], cc[3], w1, ActScale{sc.z, sc.w});
            }
        }
        if (++s == p.stages) { s = 0; ph ^= 1; }

        // combine the 16 K-slices in warp order
        float* rb = red + warp * (kMmaRows * kWideRedPitch);
#pragma unroll
        for (int j = 0; j < NT; j++) {
            *reinterpret_cast<float2*>(&rb[g * kWideRedPitch + 8 * j + 2 * tig]) = make_float2(acc[j][0], acc[j][1]);
            *reinterpret_cast<float2*>(&rb[(g + 8) * kWideRedPitch + 8 * j + 2 * tig]) = make_float2(acc[j][2], acc[j][3]);
        }
        ptx::bar_sync(1, kWideWarps * 32);
        for (int o = tid; o < kMmaRows * TOK; o += kWideWarps * 32) {
            const int row = o / TOK, tok = o - row * TOK;
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kWideWarps; w++) v += red[w * (kMmaRows * kWideRedPitch) + row * kWideRedPitch + tok];
            const int f = t * kMmaRows + row;
            if (f < p.F && tok < p.T) p.C[(int64_t)tok * p.ldc_t + (int64_t)f * p.ldc_f] = v;
        }
        __syncthreads();   // partials consumed, and every warp is done with this tile's stage:
        if (tid == 0 && t + p.stages < t_end) issue_tile(t + p.stages);   // refill it
    }
    if (p.pdl == 2) ptx::griddep_wait();
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int bigk_pitch(int wtype) {
    const int seg = kBigChunk * block_bytes(wtype);
    return seg + 16 + ((128 - (seg % 128)) % 128);
}
static size_t bigk_fixed(int nb) { return 128 + kMmaWarps * 128 * 4 + (size_t)nb * 320 + 128; }
static bool bigk_supported(int wtype, int nb) {
    return (nb % 8) == 0 && bigk_fixed(nb) + 2 * (size_t)kMmaRows * bigk_pitch(wtype) <= (size_t)kMmaSmemMax + 20 * 1024;
}
static int nbw_of(int nb) {
    const int nbw = (nb + kMmaWarps - 1) / kMmaWarps;
    return nbw <= 8 ? 8 : (nbw <= 16 ? 16 : 32);
}
static bool regs_variant_supported(int wtype, int nb) {
    if (nb < 8 || nb > kMmaWarps * 32) return false;
    const int nbw = nbw_of(nb);
    const int nc = mma_pick_nc(block_bytes(wtype), nbw);
    const int seg = (nbw / nc) * kMmaWarps * block_bytes(wtype);
    return mma_fixed(nb) + 2 * (size_t)kMmaRows * mma_pitch(seg) <= (size_t)kMmaSmemBudget;
}
bool gemv_mma_supported(int wtype, const void* act, const void* wgt, int T, int F, int K) {
    const int nb = K / 32;
    const size_t rowbytes = (size_t)nb * block_bytes(wtype);
    if (T < 1 || F < 1 || nb < 8) return false;
    if (rowbytes % 16 != 0) return false;
    if (reinterpret_cast<uintptr_t>(wgt) % 16 != 0 || reinterpret_cast<uintptr_t>(act) % 4 != 0) return false;
    return regs_variant_supported(wtype, nb) || bigk_supported(wtype, nb);
}

template <int WT>
static cudaError_t launch_bigk(const GemvMmaBigParams& p, size_t smem, int grid, bool ms_exact, cudaStream_t st) {
    auto launch = [&](auto kernel, int variant) -> cudaError_t {
        (void)variant;
        if (cudaError_t e = smem_optin(reinterpret_cast<const void*>(kernel), smem)) return e;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kMmaThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = p.pdl ? 1 : 0;
        return cudaLaunchKernelEx(&cfg, kernel, p);
    };
    cudaError_t e;
    if constexpr (Fmt<WT>::m >= 0) {
        e = ms_exact ? launch(gemv_mma_bigk_kernel<WT, true>, 1) : launch(gemv_mma_bigk_kernel<WT, false>, 0);
    } else {
        e = launch(gemv_mma_bigk_kernel<WT, false>, 0);
    }
    note_launch();
    return e;
}

template <int WT, int NBW>
static cudaError_t launch_mma_inst(const GemvMmaParams& p, size_t smem, int grid, bool ms_exact, cudaStream_t st) {
    constexpr int NC = mma_pick_nc(Fmt<WT>::bytes, NBW);
    auto launch = [&](auto kernel, int variant) -> cudaError_t {
        (void)variant;
        if (cudaError_t e = smem_optin(reinterpret_cast<const void*>(kernel), smem)) return e;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kMmaThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = p.pdl ? 1 : 0;
        return cudaLaunchKernelEx(&cfg, kernel, p);
    };
    cudaError_t e;
    const bool full = p.nb == NBW * kMmaWarps;
    if constexpr (Fmt<WT>::m >= 0) {
        if (full) e = ms_exact ? launch(gemv_mma_kernel<WT, NBW, NC, true, true>, 3) : launch(gemv_mma_kernel<WT, NBW, NC, false, true>, 2);
        else e = ms_exact ? launch(gemv_mma_kernel<WT, NBW, NC, true, false>, 1) : launch(gemv_mma_kernel<WT, NBW, NC, false, false>, 0);
    } else {
        e = full ? launch(gemv_mma_kernel<WT, NBW, NC, false, true>, 2) : launch(gemv_mma_kernel<WT, NBW, NC, false, false>, 0);
    }
    note_launch();
    return e;
}

template <int WT>
static cudaError_t launch_mma_wt(const GemvMmaParams& p, size_t smem, int grid, bool ms, cudaStream_t st) {
    const int nbw = (p.nb + kMmaWarps - 1) / kMmaWarps;
    if (nbw <= 8) return launch_mma_inst<WT, 8>(p, smem, grid, ms, st);
    if (nbw <= 16) return launch_mma_inst<WT, 16>(p, smem, grid, ms, st);
    return launch_mma_inst<WT, 32>(p, smem, grid, ms, st);
}

// wide variant: K must fill the 16 warps' fragment slots exactly (K = 4096: NBW 8, K = 8192: NBW 16)
static int wide_nbw(int nb) { return nb == 16 * 8 ? 8 : (nb == 16 * 16 ? 16 : 0); }
static size_t wide_fixed(int nb, int nt) {
    return 128 + (size_t)kWideWarps * kMmaRows * kWideRedPitch * 4 + (size_t)nb * nt * 64 + 128;
}
bool gemv_mma_wide_supported(int wtype, const void* act, const void* wgt, int T, int F, int K) {
    const int nb = K / 32, nbw = wide_nbw(nb);
    if (!nbw || T < 2 || F < 1 || block_bytes(wtype) == 0) return false;
    if (reinterpret_cast<uintptr_t>(wgt) % 16 != 0 || reinterpret_cast<uintptr_t>(act) % 4 != 0) return false;
    const int nt = nbw == 8 ? 4 : 2;
    return wide_fixed(nb, nt) + 2 * (size_t)kMmaRows * mma_pitch(nb * block_bytes(wtype)) <= (size_t)kWideSmemMax;
}

template <int WT, int NBW, int NT>
static cudaError_t launch_wide_inst(const GemvMmaWideParams& p, size_t smem, int grid, bool ms_exact, cudaStream_t st) {
    auto launch = [&](auto kernel, int variant) -> cudaError_t {
        (void)variant;
        if (cudaError_t e = smem_optin(reinterpret_cast<const void*>(kernel), smem)) return e;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kWideThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = p.pdl ? 1 : 0;
        return cudaLaunchKernelEx(&cfg, kernel, p);
    };
    cudaError_t e;
    if constexpr (Fmt<WT>::m >= 0) {
        e = ms_exact ? launch(gemv_mma_wide_kernel<WT, NBW, NT, true>, 1) : launch(gemv_mma_wide_kernel<WT, NBW, NT, false>, 0);
    } else {
        e = launch(gemv_mma_wide_kernel<WT, NBW, NT, false>, 0);
    }
    note_launch();
    return e;
}

template <int WT>
static cudaError_t launch_wide_wt(const GemvMmaWideParams& p, int nbw, int nt, size_t smem, int grid, bool ms, cudaStream_t st) {
    if (nt == 1) return nbw == 8 ? launch_wide_inst<WT, 8, 1>(p, smem, grid, ms, st) : launch_wide_inst<WT, 16, 1>(p, smem, grid, ms, st);
    if (nbw == 8) return nt == 4 ? launch_wide_inst<WT, 8, 4>(p, smem, grid, ms, st) : launch_wide_inst<WT, 8, 2>(p, smem, grid, ms, st);
    return launch_wide_inst<WT, 16, 2>(p, smem, grid, ms, st);
}

// Programmatic-dependent-launch mode of pass t0 of a multi-pass call.  QGEMM_INPUTS_READY (pdl = 2: compute at once, wait
// only before exit) applies to the FIRST pass alone; the later passes of the same call wait for their predecessor before
// they compute (pdl = 1: their weight stream still starts early).  With INPUTS_READY on every pass, three 8-token passes of
// gemv_mma_kernel computed concurrently, and in about one call in three a few weight rows of the middle pass came out wrong
// (q8_0, T = 24, K = 8192: all eight tokens of the affected rows, hundreds of times the rounding bound), while the same
// passes run one after the other were exact.
static int mma_pass_pdl(uint32_t flags, int t0) {
    if (!(flags & QGEMM_WEIGHTS_STATIC)) return 0;
    return (t0 == 0 && (flags & QGEMM_INPUTS_READY)) ? 2 : 1;
}

// T tokens in passes of 8 * NT
cudaError_t launch_gemv_mma_wide(int wtype, const void* act, const void* wgt, float* C, int T, int F, int K, int64_t ldc_t,
                                 int64_t ldc_f, uint32_t flags, int num_sms, cudaStream_t st) {
    const int nb = K / 32, nbw = wide_nbw(nb);
    if (!nbw) return cudaErrorInvalidValue;
    const int nt_max = nbw == 8 ? 4 : 2;
    const int pitch = mma_pitch(nb * block_bytes(wtype));
    const int ntiles = (F + kMmaRows - 1) / kMmaRows;
    const int grid = min(ntiles, num_sms);
    const bool ms = flags & QGEMM_MS_EXACT;
    for (int t0 = 0; t0 < T; t0 += 8 * nt_max) {
        const int tp = min(8 * nt_max, T - t0);
        const int nt = tp <= 8 ? 1 : ((nbw == 8 && tp > 16) ? 4 : 2);
        const size_t fixed = wide_fixed(nb, nt);
        int stages = (int)(((size_t)kWideSmemMax - fixed) / ((size_t)kMmaRows * pitch));
        stages = max(2, min(kMmaStagesMax, min(stages, (ntiles + grid - 1) / grid + 1)));
        GemvMmaWideParams p;
        p.act = (const uint8_t*)act + (size_t)t0 * nb * kQ81Bytes;
        p.wgt = (const uint8_t*)wgt;
        p.C = C + (int64_t)t0 * ldc_t;
        p.T = tp; p.F = F; p.nb = nb; p.ldc_t = ldc_t; p.ldc_f = ldc_f;
        p.pitch = pitch; p.stages = stages;
        p.pdl = mma_pass_pdl(flags, t0);
        const size_t smem = fixed + (size_t)stages * kMmaRows * pitch;
        cudaError_t e;
        switch (wtype) {
        case QGEMM_TYPE_Q4_0: e = launch_wide_wt<QGEMM_TYPE_Q4_0>(p, nbw, nt, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q4_1: e = launch_wide_wt<QGEMM_TYPE_Q4_1>(p, nbw, nt, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q5_0: e = launch_wide_wt<QGEMM_TYPE_Q5_0>(p, nbw, nt, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q5_1: e = launch_wide_wt<QGEMM_TYPE_Q5_1>(p, nbw, nt, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q8_0: e = launch_wide_wt<QGEMM_TYPE_Q8_0>(p, nbw, nt, smem, grid, ms, st); break;
        default: e = cudaErrorInvalidValue;
        }
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// T tokens in passes of 8
cudaError_t launch_gemv_mma(int wtype, const void* act, const void* wgt, float* C, int T, int F, int K, int64_t ldc_t,
                            int64_t ldc_f, uint32_t flags, int num_sms, cudaStream_t st, const PeerOut* peer) {
    if (peer && T > 8) return cudaErrorInvalidValue;  // peer mode: one pass per launch
    // T <= 8: the one-CTA-per-SM kernel wins only where the two-CTA one runs short of shared memory stages
    // (measured: q8_0 11008x4096 12.5 -> 11.4 us at T=8; slower for the 4-bit formats and for small matrices)
    const bool wide1 = wtype == QGEMM_TYPE_Q8_0 && (int64_t)F * K >= (1ll << 25);
    if (!peer && (T > 8 || wide1 || QGEMM_ENV("QGEMM_MMA_WIDE1")) && !QGEMM_ENV("QGEMM_MMA_NO_WIDE") &&
        gemv_mma_wide_supported(wtype, act, wgt, T, F, K))
        return launch_gemv_mma_wide(wtype, act, wgt, C, T, F, K, ldc_t, ldc_f, flags, num_sms, st);
    if (!regs_variant_supported(wtype, K / 32)) {      // long rows: fragments in smem, K-chunked stages
        const int nbk = K / 32;
        const int bp = bigk_pitch(wtype);
        const size_t fx = bigk_fixed(nbk);
        int stg = (int)(((size_t)kMmaSmemMax + 20 * 1024 - fx) / ((size_t)kMmaRows * bp));
        stg = max(2, min(kMmaStagesMax, stg));
        const int nt = (F + kMmaRows - 1) / kMmaRows;
        const int grd = min(nt, num_sms);
        const size_t sm = fx + (size_t)stg * kMmaRows * bp;
        for (int t0 = 0; t0 < T; t0 += 8) {
            GemvMmaBigParams p;
            p.act = (const uint8_t*)act + (size_t)t0 * nbk * kQ81Bytes;
            p.wgt = (const uint8_t*)wgt;
            p.C = C + (int64_t)t0 * ldc_t;
            p.T = min(8, T - t0); p.F = F; p.nb = nbk; p.ldc_t = ldc_t; p.ldc_f = ldc_f;
            p.pitch = bp; p.stages = stg;
            p.pdl = mma_pass_pdl(flags, t0);
            p.peer = peer ? *peer : PeerOut{};
            const bool ms = flags & QGEMM_MS_EXACT;
            cudaError_t e;
            switch (wtype) {
            case QGEMM_TYPE_Q4_0: e = launch_bigk<QGEMM_TYPE_Q4_0>(p, sm, grd, ms, st); break;
            case QGEMM_TYPE_Q4_1: e = launch_bigk<QGEMM_TYPE_Q4_1>(p, sm, grd, ms, st); break;
            case QGEMM_TYPE_Q5_0: e = launch_bigk<QGEMM_TYPE_Q5_0>(p, sm, grd, ms, st); break;
            case QGEMM_TYPE_Q5_1: e = launch_bigk<QGEMM_TYPE_Q5_1>(p, sm, grd, ms, st); break;
            case QGEMM_TYPE_Q8_0: e = launch_bigk<QGEMM_TYPE_Q8_0>(p, sm, grd, ms, st); break;
            default: e = cudaErrorInvalidValue;
            }
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    const int nb = K / 32;
    const int nbw = nbw_of(nb);
    const int nc = mma_pick_nc(block_bytes(wtype), nbw);
    const int cb = (nbw / nc) * kMmaWarps;                 // blocks per chunk
    const int pitch = mma_pitch(cb * block_bytes(wtype));
    const size_t fixed = mma_fixed(nb);
    int stages = (int)(((size_t)kMmaSmemBudget - fixed) / ((size_t)kMmaRows * pitch));
    stages = max(2, min(kMmaStagesMax, stages));
    if (const char* e = QGEMM_ENV("QGEMM_MMA_STAGES")) stages = max(2, min(stages, atoi(e)));  // tuning aid
    const int span = QGEMM_ENV("QGEMM_MMA_SPAN") ? 1 : 0;
    const int ntiles = (F + kMmaRows - 1) / kMmaRows;
    const int grid = span ? min(F, 2 * num_sms) : min(ntiles, 2 * num_sms);
    const int chunks_per_cta = (span ? ((F + grid - 1) / grid + kMmaRows - 1) / kMmaRows : (ntiles + grid - 1) / grid) * ((nb + cb - 1) / cb);
    stages = max(2, min(stages, chunks_per_cta));
    const size_t smem = fixed + (size_t)stages * kMmaRows * pitch;
    for (int t0 = 0; t0 < T; t0 += 8) {
        GemvMmaParams p;
        p.act = (const uint8_t*)act + (size_t)t0 * nb * kQ81Bytes;
        p.wgt = (const uint8_t*)wgt;
        p.C = C + (int64_t)t0 * ldc_t;
        p.T = min(8, T - t0); p.F = F; p.nb = nb; p.ldc_t = ldc_t; p.ldc_f = ldc_f;
        p.pitch = pitch; p.stages = stages; p.span = span; p.pdl = mma_pass_pdl(flags, t0);
        p.peer = peer ? *peer : PeerOut{};
        const bool ms = flags & QGEMM_MS_EXACT;
        cudaError_t e;
        switch (wtype) {
        case QGEMM_TYPE_Q4_0: e = launch_mma_wt<QGEMM_TYPE_Q4_0>(p, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q4_1: e = launch_mma_wt<QGEMM_TYPE_Q4_1>(p, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q5_0: e = launch_mma_wt<QGEMM_TYPE_Q5_0>(p, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q5_1: e = launch_mma_wt<QGEMM_TYPE_Q5_1>(p, smem, grid, ms, st); break;
        case QGEMM_TYPE_Q8_0: e = launch_mma_wt<QGEMM_TYPE_Q8_0>(p, smem, grid, ms, st); break;
        default: e = cudaErrorInvalidValue;
        }
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace qgemm
