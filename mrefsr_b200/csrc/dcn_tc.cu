// mrefsr_b200/csrc/dcn_tc.cu -- DCNv2 forward on tcgen05 (TF32 operands, fp32 accumulation in TMEM).
//
// Replaces the reference's per-sample {im2col kernel -> columns buffer in HBM -> cuBLAS addmm_}
// (basicsr/ops/dcn/src/deform_conv_cuda.cpp:539-555, deform_conv_cuda_kernel.cu:571-633) with ONE launch of
// dcn_tc_split_kernel over the whole batch in which the deformable im2col tile never leaves the SM.
//
//   CTA tile   : 256 output positions x all Co output channels.  The 256 rows are square-ish patches of positions
//                (16x16, or four 8x8 for small grids) so that the bilinear corners of x- and y-neighbours meet
//                in L1 within one K step; grids that would need > 3 % padding rows use 256 consecutive positions
//                of the B*Ho*Wo concatenation instead.
//   K loop     : (32-channel slab) x (tap).  Per step the A tile [256 x 32] fp32 is produced on the SM by the
//                producer warps and stored straight into 128B-swizzled shared memory; the B tile [Co x 32] of the
//                repacked (tf32-rounded) weights arrives by TMA; one elected thread of the MMA warp issues
//                2 (M halves) x 4 (K = 8 steps) tcgen05.mma.kind::tf32 into TMEM.
//   warp roles : (a) 8 decode warps, thread = tile row, fill a shared-memory sample table ahead of the gather -- per
//                (row, deform group): corner offset into an NHWC copy of the input + the four bilinear weights with
//                mask and corner validity folded in -- from position-major (coalesced) offset / mask reads issued
//                two tables earlier;
//                (b) 16 gather warps, as two groups of eight on alternate K steps: per (row, 8-channel chunk) four
//                256-bit corner loads, blend, round to tf32, two 16-byte swizzled stores;
//                (c) one MMA warp.  All hand-offs are mbarriers with ONE elected arrive per warp (table ring
//                full/empty, stage ring full/empty); there is no CTA-wide barrier in the loop.
//   epilogue   : gather warps 0..3 and 8..11 also drain finished accumulators (tcgen05.ld 32x32b, bias add,
//                position-major coalesced NCHW stores); they poll the TMEM-full barrier while they wait.
//
// Why the roles are split (profiles/r01_dcn_gather_microbench.txt, r01s_dcn_ab.md, r01u_dcn_tc_split_ncu_full.txt):
// the bilinear gather alone needs 0.35 / 0.79 / 2.07 ms per 80-sample call with 64 warps/SM -- about one 32-byte
// sector per clock per SM through L1.  A kernel whose 17 warps each decoded AND gathered took 0.73 / 1.26 / 2.74 ms:
// latency bound inside the producer loop, not bandwidth bound -- 96 registers each (one SM sub-partition hosts 5 of
// them), a serial chain of ~440 instructions and two dependent memory round trips per K step; raising the L1 hit rate
// from 45 % to 65 % (2-D patches), halving the gathered bytes (fp16 staging) or keeping the offset stream out of L1
// each bought 2-4 %, and more loads in flight per warp cost 15-20 %.  With decode and gather on different warps
// (25 warps, 72 registers) the round-1 kernel took 0.56 / 0.99 / 2.22 ms: 0.93 sectors/clk/SM at the large scale,
// i.e. at the gather's own ceiling.  The K loops are kept lean: no integer division, per-tile row state, 8-channel
// gather items (one 256-bit load per corner, packed fp32x2 FMAs).
// Tried and rejected on B200: separate table warps at 17 warps, register-resident decode, a group-major
// zero-bordered layout, two 128-row CTAs per SM, a 16-warp CTA whose last-arriving warp issues the MMAs (128
// registers, two items in flight), corner fetch by TMA tile::gather4 (10 clk per gather4 per SM: 5 ms at the large
// scale), an fp16 2x2-packed corner layout, an fp16 NHWC staging copy with a device-side range gate (-2 %),
// cp.async.bulk.prefetch.L2 of the input, deeper stage rings at the expense of L1 (+8 %), the table decode moved
// under the corner loads' latency (spills at the register cap: +16 %), cp.async staging of the raw offsets (+5 %).
//
// Round 2 (profiles/r02_dcn_window.md): an ablation of dcn_tc_split_kernel showed that its parts -- pipeline skeleton,
// decode, gather, epilogue stores, MMAs -- add up almost serially and that a FREE corner fetch would save only a fifth of
// its time, i.e. the kernel is bound by instruction issue and hand-off latency, not by the L1 sector rate.  The gather
// warps therefore no longer walk every K step in lock-step: they work as two groups of eight on alternate K steps, a
// third pipeline stage is used where a deform group has >= 16 channels, and the decode handles interior sampling
// points without clamps / validity bits: 0.55 / 0.88 / 1.96 ms per launch, same bits.  A second corner fetch that
// staged each patch's input window in shared memory by TMA gave the same bits and was slower on every flow kind
// (same profile); it was removed (DESIGN.md 2.2b).
//
// The 3-pass mode (MREFSR_DCN_TF32X3 / the MREFSR_DCN_X3 flag, X3 = true instantiations) keeps this geometry and halves
// the channels per K step: each 128-byte row holds the tf32 hi AND lo parts of 16 channels, and the MMA warp issues
// lo.hi + hi.lo + hi.hi, which gives fp32-grade results at the price of twice the K steps (DESIGN.md 2.2).
//
// Offsets / masks come either as materialised tensors (the reference operator API) or -- fused DynAgg mode --
// straight from the raw conv_offset_mask output plus the matcher's arg-max map: offset = conv + s*flow shifted
// by the tap, mask = sigmoid(conv) (basicsr/archs/ref_mrapa_restoration_arch.py:55-68 and
// corres_generation_arch.py:70-105 folded into the gather), which removes two full passes over the
// 216-plane tensor.
#include <stdlib.h>
#include "dcn_tc.cuh"
#include "../../include/mrefsr_b200.h"

namespace mrefsr {


// NCHW -> NHWC (fp32): tile = 32 pixels x up to 128 channels per CTA (256 threads).  Loads: lane = pixel (128-byte
// coalesced, 16 independent loads per thread in flight); stores: one float4 (4 channels) per lane, 512 bytes
// contiguous per warp.  grid (ceil(HW/32), ceil(C/128), B)
template <bool ROUND,      // ROUND: values rounded to tf32 on the way (operands of the tcgen05 GEMMs, whose reads truncate)
          bool SPLIT = false>   // SPLIT (with ROUND): dst gets tf32(v), dst_lo tf32(v - tf32(v)) (3-pass GEMM operands)
__global__ void __launch_bounds__(256)
nchw_to_nhwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW, float* __restrict__ dst_lo) {
    __shared__ float tile[128][33];
    const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 128;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* s = src + (size_t)b * C * HW;
    float* d = dst + (size_t)b * C * HW;
    const int p = p0 + lane;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int cl = warp + 8 * i, c = c0 + cl;
        const float v = (c < C && p < HW) ? __ldcs(s + (size_t)c * HW + p) : 0.f;
        tile[cl][lane] = (ROUND && !SPLIT) ? to_tf32(v) : v;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int pl = warp * 4 + j, pp = p0 + pl, c = c0 + lane * 4;
        if (pp < HW && c < C) {   // C % 4 == 0 on this path (C % 32 == 0 is an eligibility condition)
            const float4 v = make_float4(tile[lane * 4][pl], tile[lane * 4 + 1][pl], tile[lane * 4 + 2][pl],
                                         tile[lane * 4 + 3][pl]);
            if (SPLIT) {
                const float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
                *reinterpret_cast<float4*>(d + (size_t)pp * C + c) = h;
                *reinterpret_cast<float4*>(dst_lo + (size_t)b * C * HW + (size_t)pp * C + c) =
                    make_float4(to_tf32(v.x - h.x), to_tf32(v.y - h.y), to_tf32(v.z - h.z), to_tf32(v.w - h.w));
            } else {
                *reinterpret_cast<float4*>(d + (size_t)pp * C + c) = v;
            }
        }
    }
}

// W[co][c][tap] -> Wt[co][tap*C + c], rounded to tf32 (round-to-nearest, so the MMA's operand truncation is exact)
__global__ void dcn_weight_repack_kernel(const float* __restrict__ w, float* __restrict__ wt, int Co, int C, int K) {
    const int total = Co * C * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int c = i % C, tap = (i / C) % K, co = i / (C * K);
        wt[i] = to_tf32(__ldg(w + ((size_t)co * C + c) * K + tap));
    }
}

// W[co][c][tap] -> Wt[co][tap][C/16][hi c0..7 | hi c8..15 | lo c0..7 | lo c8..15]: the B operand of the 3-pass kernels,
// one 128-byte TMA row per 16-channel slab (hi = tf32(w), lo = tf32(w - hi); cvt.rna clears the low bits)
__global__ void dcn_weight_repack_x3_kernel(const float* __restrict__ w, float* __restrict__ wt, int Co, int C, int K) {
    const int total = Co * C * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int c = i % C, tap = (i / C) % K, co = i / (C * K);
        const float v = __ldg(w + ((size_t)co * C + c) * K + tap), hi = to_tf32(v);
        float* o = wt + ((size_t)co * K + tap) * 2 * C + (c / TBK_X3) * 2 * TBK_X3 + c % TBK_X3;
        o[0] = hi;
        o[TBK_X3] = to_tf32(v - hi);
    }
}


// Drain M halves [half_lo, half_hi) of one finished accumulator tile: tcgen05.ld 32x32b, bias add, position-major
// coalesced NCHW stores.
__device__ __forceinline__ void dcn_epilogue_tile(const DcnTcParams& prm, const float* __restrict__ bias,
                                                  uint32_t tmem_base, uint64_t* tempty_bar, int tile, int buf, int warp,
                                                  int lane, int half_lo, int half_hi) {
    const int Co = prm.s.Co, P = prm.P;
#pragma unroll 1
    for (int half = half_lo; half < half_hi; ++half) {
        int b = 0, oy = 0, ox = 0;
        const bool ok = dcn_row_coords(prm, tile, half * 128 + warp * 32 + lane, b, oy, ox);
        const int p = ok ? oy * prm.s.Wo + ox : 0;
        if (!ok) b = 0;
        const int bd = prm.dst_group ? (b / prm.dst_group) * prm.dst_stride + prm.dst_offset + b % prm.dst_group : b;
        int k_lo = 0, k_hi = prm.n_outs, Pd = P;      // destination buffers of this row, plane size there
        size_t o_off = prm.out_nhwc ? ((size_t)bd * P + p) * Co : (size_t)bd * Co * P + p;
        if (prm.dst_slab_rows) {
            k_lo = oy / prm.dst_slab_rows;
            k_hi = k_lo + 1;
            Pd = prm.dst_slab_rows * prm.s.Wo;
            o_off = (size_t)bd * Co * Pd + (size_t)(oy - k_lo * prm.dst_slab_rows) * prm.s.Wo + ox;
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + buf * 2 * Co + half * Co;
#pragma unroll 1
        for (int c0 = 0; c0 < Co; c0 += 8) {
            uint32_t v[8];
            tmem_ld_32x8(taddr + c0, v);
            tmem_ld_wait();
#ifdef MREFSR_DCN_DEBUG
            if (prm.dbg & 16) continue;              // ablation 16: no epilogue stores
#endif
            if (ok) {
                float f[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    f[e] = __uint_as_float(v[e]) + (bias ? __ldg(bias + c0 + e) : 0.f);
                    f[e] = f[e] > 0.f ? f[e] : f[e] * prm.out_slope;
                }
#pragma unroll 1
                for (int k = k_lo; k < k_hi; ++k) {
                    float* o = prm.outs[k] + o_off;
                    if (prm.out_nhwc) {        // 32 contiguous bytes per thread: one full sector
                        *reinterpret_cast<float4*>(o + c0) = make_float4(f[0], f[1], f[2], f[3]);
                        *reinterpret_cast<float4*>(o + c0 + 4) = make_float4(f[4], f[5], f[6], f[7]);
                    } else {               // position-major: 32 lanes = 32 consecutive positions of one channel plane
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[(size_t)(c0 + e) * Pd] = f[e];
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tempty_bar);
}

// MMA issuer (one elected thread of the MMA warp): per tile wait for a free TMEM accumulator, per K step wait for the
// A / B stage, issue 2 (M halves) x 4 (K = 8) tcgen05.mma.kind::tf32, release the stage with a commit; a last commit
// hands the accumulator to the epilogue warps.
// X3: the stage holds [hi 16 | lo 16] channels of A and B; per M half and 8-channel step kk in {0, 1}: lo.hi, hi.lo,
// hi.hi into the same accumulator (6 MMAs per 16 channels).
template <bool X3>
__device__ __forceinline__ void dcn_mma_issuer(const DcnTcParams& prm, uint8_t* smem, uint64_t* full, uint64_t* empty,
                                               uint64_t* tfull, uint64_t* tempty, uint32_t tmem_base, int nkb_tile) {
    const int Co = prm.s.Co, S = prm.stages;
    const uint32_t idesc = umma_idesc(2, 128, Co);
    int stage = 0, it = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < prm.tiles; tile += gridDim.x, ++it) {
        const int buf = it & (prm.nbuf - 1);
        const uint32_t bphase = (it >> (prm.nbuf - 1)) & 1;
        mbar_wait_backoff(&tempty[buf], bphase ^ 1, 32);
        tc_fence_after();
        const uint32_t tacc = tmem_base + buf * 2 * Co;
        uint32_t accumulate = 0;
        for (int kb = 0; kb < nkb_tile; ++kb) {
            mbar_wait_backoff(&full[stage], phase, 20);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + (size_t)stage * prm.stage_bytes);
            const uint32_t sb = sa + T_A_BYTES;
            if (X3) {
#pragma unroll
                for (int kk = 0; kk < 2; ++kk) {
#ifdef MREFSR_DCN_DEBUG
                    if (prm.dbg & 8) continue;
#endif
                    const uint64_t bh = umma_desc_sw128(sb + kk * 32, 0), bl = umma_desc_sw128(sb + (kk + 2) * 32, 0);
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        const uint32_t ah = sa + half * (128 * 128) + kk * 32;
                        umma_tf32(tacc + half * Co, umma_desc_sw128(ah + 64, 0), bh, idesc, accumulate);
                        umma_tf32(tacc + half * Co, umma_desc_sw128(ah, 0), bl, idesc, 1);
                        umma_tf32(tacc + half * Co, umma_desc_sw128(ah, 0), bh, idesc, 1);
                    }
                    accumulate = 1;
                }
            } else {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
#ifdef MREFSR_DCN_DEBUG
                    if (prm.dbg & 8) continue;           // ablation 8: no MMAs
#endif
                    const uint64_t db = umma_desc_sw128(sb + kk * 32, 0);
                    umma_tf32(tacc, umma_desc_sw128(sa + kk * 32, 0), db, idesc, accumulate);
                    umma_tf32(tacc + Co, umma_desc_sw128(sa + 128 * 128 + kk * 32, 0), db, idesc, accumulate);
                    accumulate = 1;
                }
            }
            umma_commit(&empty[stage]);
            if (++stage == S) {
                stage = 0;
                phase ^= 1;
            }
        }
        umma_commit(&tfull[buf]);
    }
}

// ---------------------------------------------------------------------------------------------------------
// dcn_tc_split_kernel: the producer work divided between 16 gather warps (table read, corner loads, blend, swizzled
// store; warps 0..3 and 8..11 also drain TMEM while they wait) and 8 decode warps (thread = tile row: raw offset /
// mask loads two tables ahead in two register sets, branch-free sample-table decode whose GS entries per row are
// independent chains), plus the MMA warp: 25 warps under a 72-register cap.  Ring slot and phase are derived from
// the K-step index.  Measured on B200 (profiles/r01s_dcn_ab.md) against 17 warps under 96 registers that each
// decoded AND gathered: 4.81 -> 3.77 ms per step (0.56 / 0.99 / 2.21 ms per launch), same bits.  Staging the raw
// words in shared memory with cp.async instead of registers (2-4 tables ahead, no spills) was 3-6 % slower.
constexpr int S_GW = 16;                            // gather warps (threads 0..511)
constexpr int S_DW = 8;                             // decode warps (threads 512..767), one thread per tile row
constexpr int S_MMA_WARP = S_GW + S_DW;
constexpr int S_THREADS = (S_GW + S_DW + 1) * 32;   // 800
#ifndef MREFSR_S_NTAB
#define MREFSR_S_NTAB 4
#endif
constexpr int S_NTAB = MREFSR_S_NTAB;               // sample-table ring depth (decode warps run up to this far ahead)
static_assert((S_NTAB & (S_NTAB - 1)) == 0, "ring slot and phase are derived from the K-step index");

template <int GS>
struct DcnRaw {                                     // inputs of one table row (one tap, GS deform groups)
    float dy[GS], dx[GS], mk[GS];
    int mi, fyx;
};

// The gather warps work as two groups of eight that take alternate K steps (256 threads cover the 256 rows x 4 chunks
// of a K step with four items each) instead of all sixteen walking every K step in lock-step: while one group waits
// for its stage to be consumed, the other gathers.  Same arithmetic, same bits; measured on B200 (profiles/r02x):
// 3.72 -> 3.36 ms per step on coherent flows, and with the groups decoupled a third stage pays at 16+ channels per
// deform group (mid scale 0.93 -> 0.84 ms).
//
// X3 (3-pass split-tf32, fp32-grade): same stage geometry, but a K step covers a 16-channel slab whose 128-byte rows
// are [hi c0..7 | hi c8..15 | lo c0..7 | lo c8..15]; a gather thread then owns two (row, 8-channel chunk) items per
// K step instead of four, the MMA warp issues lo.hi + hi.lo + hi.hi, and the weights come packed the same way
// (dcn_weight_repack_x3_kernel).  The stage bytes, stage count and TMEM use are those of the tf32 kernel.
template <bool FUSED, int GS,       // GS = deform groups per slab (prm.gs: 1, 2 or 4; X3: 1 or 2)
          bool X3 = false>
__global__ void __launch_bounds__(S_THREADS, 1)
dcn_tc_split_kernel(const __grid_constant__ CUtensorMap mapW, const float* __restrict__ xt,
                    const float* __restrict__ offset, const float* __restrict__ mask,
                    const long long* __restrict__ max_idx, const float* __restrict__ bias,
                    const __grid_constant__ DcnTcParams prm) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    const DcnShape& s = prm.s;
    const int S = prm.stages;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)S * prm.stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + S;
    uint64_t* tfull = bars + 2 * S;
    uint64_t* tempty = tfull + 2;
    uint64_t* tab_full = tempty + 2;          // [S_NTAB]
    uint64_t* tab_empty = tab_full + S_NTAB;  // [S_NTAB]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tab_empty + S_NTAB);
    constexpr int tab_n = GS * TAB_STRIDE;      // compile-time: table addresses are register + immediate
    int* tab_base = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(bars) + 256);
    float* tab_w = reinterpret_cast<float*>(tab_base + S_NTAB * tab_n);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int Co = s.Co, C = s.C, K = prm.taps, P = prm.P;
    const int nkb_tile = prm.n_slabs * K;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&mapW);
        for (int i = 0; i < S; ++i) {
            mbar_init(&full[i], S_GW / 2 + 1);   // one elected arrive per gather warp of a group + the TMA expect_tx arrive
            mbar_init(&empty[i], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 8);
        }
        for (int a = 0; a < S_NTAB; ++a) {
            mbar_init(&tab_full[a], S_DW);
            mbar_init(&tab_empty[a], S_GW / 2);
        }
        fence_mbar_init();
    }
    if (warp == S_MMA_WARP) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int my_tiles = (prm.tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int total_kb = my_tiles * nkb_tile;   // K steps of this CTA, flattened over its tiles: (tile, slab, tap)

    if (warp < S_GW) {
        // ------------------------------------------------------------------ gather warps, two groups on alternate K steps
        constexpr int SLAB = X3 ? TBK_X3 : TBK;    // channels per K step
        constexpr int ITEMS = X3 ? 2 : 4;          // (row, 8-channel chunk) items per thread and K step
        constexpr int RSTEP = TBM / ITEMS;         // row distance between a thread's items
        const int grp = warp >> 3;                 // this group's K steps: kb = grp (mod 2)
        const int tg = threadIdx.x & 255;          // thread within the group
        const int ch = tg & (SLAB / 8 - 1);        // 8-channel chunk within the slab
        const int r0 = tg >> (X3 ? 1 : 2);         // rows r0 + RSTEP i, i < ITEMS
        const int gsub = (ch * 8) / prm.cdg;
        const uint32_t a_off0 = (uint32_t)r0 * 128u + (uint32_t)(((2 * ch) ^ (r0 & 7)) << 4);
        const uint32_t a_off1 = (uint32_t)r0 * 128u + (uint32_t)(((2 * ch + 1) ^ (r0 & 7)) << 4);
        // X3: the lo halves of the chunk go to 16-byte chunks 2ch + 4, 2ch + 5 of the row
        const uint32_t a_off2 = (uint32_t)r0 * 128u + (uint32_t)(((2 * ch + 4) ^ (r0 & 7)) << 4);
        const uint32_t a_off3 = (uint32_t)r0 * 128u + (uint32_t)(((2 * ch + 5) ^ (r0 & 7)) << 4);
        // epilogue duty: warps 0..3 drain rows 0..127 of a tile, warps 8..11 rows 128..255 (TMEM lane quarter = warp % 4)
        const bool is_epi = (warp & 7) < 4;
        int ep_done = 0, prod_done = 0;
        const int nbuf_mask = prm.nbuf - 1;
        auto poll_epilogue = [&]() {
            if (is_epi && ep_done < prod_done) {
                const int buf = ep_done & nbuf_mask;
                if (mbar_try_wait(&tfull[buf], (ep_done >> nbuf_mask) & 1)) {
                    tc_fence_after();
                    dcn_epilogue_tile(prm, bias, tmem_base, &tempty[buf], (int)blockIdx.x + ep_done * (int)gridDim.x, buf,
                                      warp & 3, lane, grp, grp + 1);
                    ++ep_done;
                }
            }
        };
        auto wait_poll = [&](uint64_t* bar, uint32_t parity) {
            // (a nanosleep back-off between polls -- 20 / 50 / 100 ns -- changes nothing: measured, profiles/r02_dcn_window.md)
            while (!mbar_try_wait(bar, parity)) poll_epilogue();
        };
        int stage = grp % S, c_slab = 0, c_tap = grp;
        uint32_t phase = 0;
        while (c_tap >= K) {                       // (K = 1 kernels)
            c_tap -= K;
            if (++c_slab == prm.n_slabs) {
                c_slab = 0;
                ++prod_done;
            }
        }
        const int dx_elems = C, dy_elems = s.W * C;
        for (int kb = grp; kb < total_kb; kb += 2) {
            const int g_slot = kb & (S_NTAB - 1);
            const uint32_t g_phase = (uint32_t)(kb / S_NTAB) & 1u;
            poll_epilogue();
            const float* xs = xt + (c_slab * SLAB + ch * 8);
            const int* tb = tab_base + g_slot * tab_n + gsub * TAB_STRIDE + r0;
            const float* tw = tab_w + g_slot * 4 * tab_n + gsub * TAB_STRIDE + r0;
            wait_poll(&tab_full[g_slot], g_phase);
            wait_poll(&empty[stage], phase ^ 1);
            uint8_t* A = smem + (size_t)stage * prm.stage_bytes;
            if (tg == 0) {        // weight tile of this K step (TMA, lands on the same full barrier)
                mbar_expect_tx(&full[stage], Co * 128);
                // (X3: a tap's packed row is 2C floats, one 32-float block per 16-channel slab)
                tma_load_3d(A + T_A_BYTES, &mapW, &full[stage], c_tap * (X3 ? 2 * C : C) + c_slab * TBK, 0, 0);
            }
#pragma unroll 1
            for (int pr = 0; pr < ITEMS / 2; ++pr) {
#pragma unroll
                for (int ii = 0; ii < 2; ++ii) {
                    const int i = pr * 2 + ii;
                    const int r = RSTEP * i;
                    const int bf = tb[r];
                    const float w0 = tw[r], w1 = tw[r + tab_n], w2 = tw[r + 2 * tab_n], w3 = tw[r + 3 * tab_n];
                    const unsigned i0 = (unsigned)(bf & ~3);
                    const unsigned i1 = i0 + ((bf & 1) ? dx_elems : 0);
                    const unsigned i2 = i0 + ((bf & 2) ? dy_elems : 0);
                    const unsigned i3 = i2 + ((bf & 1) ? dx_elems : 0);
                    const F8 v0 = ldg8(xs + i0), v1 = ldg8(xs + i1), v2 = ldg8(xs + i2), v3 = ldg8(xs + i3);
                    const float2 p0 = make_float2(w0, w0), p1 = make_float2(w1, w1), p2 = make_float2(w2, w2),
                                 p3 = make_float2(w3, w3);
                    float2 o[4], ol[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float2 a = __fmul2_rn(p0, v0.v[e]);
                        a = __ffma2_rn(p1, v1.v[e], a);
                        a = __ffma2_rn(p2, v2.v[e], a);
                        a = __ffma2_rn(p3, v3.v[e], a);
                        if (X3) {
                            tf32_split_bits(a.x, o[e].x, ol[e].x);
                            tf32_split_bits(a.y, o[e].y, ol[e].y);
                        } else {
                            o[e] = make_float2(tf32_round_bits(a.x), tf32_round_bits(a.y));
                        }
                    }
                    *reinterpret_cast<float4*>(A + a_off0 + i * (RSTEP * 128)) = make_float4(o[0].x, o[0].y, o[1].x, o[1].y);
                    *reinterpret_cast<float4*>(A + a_off1 + i * (RSTEP * 128)) = make_float4(o[2].x, o[2].y, o[3].x, o[3].y);
                    if (X3) {
                        *reinterpret_cast<float4*>(A + a_off2 + i * (RSTEP * 128)) =
                            make_float4(ol[0].x, ol[0].y, ol[1].x, ol[1].y);
                        *reinterpret_cast<float4*>(A + a_off3 + i * (RSTEP * 128)) =
                            make_float4(ol[2].x, ol[2].y, ol[3].x, ol[3].y);
                    }
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&full[stage]);
                mbar_arrive(&tab_empty[g_slot]);
            }
            stage += 2;
            if (stage >= S) {
                stage -= S;
                phase ^= 1;
            }
            c_tap += 2;
            while (c_tap >= K) {
                c_tap -= K;
                if (++c_slab == prm.n_slabs) {
                    c_slab = 0;
                    ++prod_done;      // this group has produced all of its K steps of the tile
                }
            }
        }
        prod_done = my_tiles;
        while (is_epi && ep_done < prod_done) {    // drain the remaining accumulators
            const int buf = ep_done & nbuf_mask;
            mbar_wait_backoff(&tfull[buf], (ep_done >> nbuf_mask) & 1, 64);
            tc_fence_after();
            dcn_epilogue_tile(prm, bias, tmem_base, &tempty[buf], (int)blockIdx.x + ep_done * (int)gridDim.x, buf, warp & 3,
                              lane, grp, grp + 1);
            ++ep_done;
        }
    } else if (warp < S_MMA_WARP) {
        // ------------------------------------------------------------------ decode warps
        const int erow = threadIdx.x - S_GW * 32;  // tile row owned by this thread
        // ---- per-tile state of this thread's row, load cursor
        int l_tile = blockIdx.x, l_slab = 0, l_tap = 0, l_dg0 = 0;
        const unsigned kw_magic = 65536u / (unsigned)s.kw + 1u;      // tap / kw == (tap * kw_magic) >> 16 for tap < 256
        int row_yx = -1, row_bH = 0, row_qyx = 0, row_idx0 = 0;
        const float* row_off = offset;
        const float* row_msk = mask;
        auto decode_rows = [&](int tile) {
            int b = 0, oy = 0, ox = 0;
            row_yx = -1;
            if (dcn_row_coords(prm, tile, erow, b, oy, ox)) {
                const int p = oy * s.Wo + ox;
                row_yx = (oy << 16) | ox;
                row_bH = b * s.H;
                if (FUSED) {
                    row_off = offset + (size_t)b * 3 * s.DG * K * P + p;
                    row_qyx = ((oy / prm.flow_scale) << 16) | (ox / prm.flow_scale);
                    row_idx0 = b * prm.hp * prm.wp;
                } else {
                    row_off = offset + (size_t)b * 2 * s.DG * K * P + p;
                    if (mask) row_msk = mask + (size_t)b * s.DG * K * P + p;
                }
            }
        };
        // the row coordinates travel with the raw inputs: a table loaded for the next tile is decoded after
        // decode_rows has already moved this thread to that tile, but one loaded for the LAST step of a tile must be
        // decoded with that tile's coordinates -> keep (yx, bH) per raw set
        struct RawRow {
            DcnRaw<GS> r;
            int yx, bH;
        };
        auto load_next = [&](RawRow& rr, int l_kb) {      // rr <- inputs of table l_kb, then advance the load cursor
            rr.yx = row_yx;
            rr.bH = row_bH;
            rr.r.fyx = -1;
#ifdef MREFSR_DCN_DEBUG
            if (row_yx >= 0 && !(prm.dbg & 2)) {     // ablation 2: no offset / mask loads
#else
            if (row_yx >= 0) {
#endif
#pragma unroll
                for (int g = 0; g < GS; ++g) {
                    {
                        const int dgi = l_dg0 + g;
                        if (!FUSED) {
                            const unsigned o = (unsigned)((dgi * 2 * K + 2 * l_tap) * P);
                            rr.r.dy[g] = ldg_early(row_off + o);
                            rr.r.dx[g] = ldg_early(row_off + o + (unsigned)P);
                            rr.r.mk[g] = mask ? ldg_early(row_msk + (unsigned)((dgi * K + l_tap) * P)) : 1.f;
                        } else {
                            const unsigned o = (unsigned)(2 * (dgi * K + l_tap) * P);
                            rr.r.dy[g] = ldg_early(row_off + o);
                            rr.r.dx[g] = ldg_early(row_off + o + (unsigned)P);
                            rr.r.mk[g] = ldg_early(row_off + (unsigned)((2 * s.DG * K + dgi * K + l_tap) * P));
                        }
                    }
                }
                if (FUSED) {
                    const int l_ti = (int)(((unsigned)l_tap * kw_magic) >> 16), l_tj = l_tap - l_ti * s.kw;
                    const int fy = (row_qyx >> 16) - l_ti, fx = (row_qyx & 0xffff) - l_tj;
                    if (fy >= 0 && fx >= 0 && fy < prm.hp && fx < prm.wp) {
                        rr.r.mi = ldg_early_s32(reinterpret_cast<const int*>(max_idx + (row_idx0 + fy * prm.wp + fx)));
                        rr.r.fyx = (fy << 16) | fx;
                    }
                }
            }
            if (++l_tap == K) {
                l_tap = 0;
                if (++l_slab == prm.n_slabs) {
                    l_slab = 0;
                    l_tile += gridDim.x;
                    if (l_kb + 1 < total_kb) decode_rows(l_tile);
                }
                constexpr int SLAB = X3 ? TBK_X3 : TBK;
                l_dg0 = (prm.cdg >= SLAB) ? (l_slab * SLAB) / prm.cdg : l_slab * (SLAB / prm.cdg);
            }
        };
        int d_tap = 0;                                           // tap of the table being decoded
        auto decode_store = [&](const RawRow& rr, int d_kb) {   // rr = inputs of table d_kb -> its ring slot
            const int d_slot = d_kb & (S_NTAB - 1);
            const uint32_t d_phase = (uint32_t)(d_kb / S_NTAB) & 1u;
            mbar_wait(&tab_empty[d_slot], d_phase ^ 1);
            int* tb = tab_base + d_slot * tab_n + erow;
            float* tw = tab_w + d_slot * 4 * tab_n + erow;
            float ybase = 0.f, xbase = 0.f, fly = 0.f, flx = 0.f;
            if (rr.yx >= 0) {
                const int d_ti = (int)(((unsigned)d_tap * kw_magic) >> 16), d_tj = d_tap - d_ti * s.kw;
                ybase = (float)((rr.yx >> 16) * s.sh - s.ph + d_ti * s.dh);
                xbase = (float)((rr.yx & 0xffff) * s.sw - s.pw + d_tj * s.dw);
                if (FUSED && rr.r.fyx >= 0) {
                    const int my = (int)__umulhi((unsigned)rr.r.mi, prm.wp_magic), mx = rr.r.mi - my * prm.wp;
                    fly = (float)((my - (rr.r.fyx >> 16)) * prm.flow_scale);
                    flx = (float)((mx - (rr.r.fyx & 0xffff)) * prm.flow_scale);
                }
            }
            // Branch-free per entry (everything is computed and then selected), so that the up-to-four entries of a
            // row are independent straight-line chains the scheduler can interleave.
            const bool row_ok = rr.yx >= 0;
#ifdef MREFSR_DCN_DEBUG
            if (prm.dbg & 4) {                       // ablation 4: no sample decode (constant table entries)
#pragma unroll
                for (int g = 0; g < GS; ++g) {
                    const int e = g * TAB_STRIDE;
                    tb[e] = 0;
                    tw[e] = tw[e + tab_n] = tw[e + 2 * tab_n] = tw[e + 3 * tab_n] = 0.25f;
                }
            } else
#endif
#pragma unroll
            for (int g = 0; g < GS; ++g) {
                {
                    const float y = ybase + (FUSED ? rr.r.dy[g] + fly : rr.r.dy[g]);
                    const float x = xbase + (FUSED ? rr.r.dx[g] + flx : rr.r.dx[g]);
                    const bool in = row_ok && y > -1.f && x > -1.f && y < (float)s.H && x < (float)s.W;
                    const float mk = FUSED ? __fdividef(1.f, 1.f + __expf(-rr.r.mk[g])) : rr.r.mk[g];
                    const float fy0 = floorf(y), fx0 = floorf(x);
                    const int y0 = (int)fy0, x0 = (int)fx0;       // saturating conversions: garbage in, garbage selected away
                    const float ly = y - fy0, lx = x - fx0, hy = 1.f - ly, hx = 1.f - lx;
                    const float hym = hy * mk, lym = ly * mk;
                    // Interior sampling points (all four corners inside the plane: everything but the outermost ring)
                    // need no clamping and no validity bits; the border rule is a rarely taken fix-up.  Same values
                    // as the one-formula version bit for bit, ~16 instructions fewer per entry on the common path.
                    int base = (((rr.bH + y0) * s.W + x0) * C) | 3;
                    float w0 = hym * hx, w1 = hym * lx, w2 = lym * hx, w3 = lym * lx;
                    if (in && !((unsigned)y0 < (unsigned)(s.H - 1) && (unsigned)x0 < (unsigned)(s.W - 1))) {
                        const bool ty0 = y0 >= 0, ty1 = y0 <= s.H - 2, tx0 = x0 >= 0, tx1 = x0 <= s.W - 2;
                        const int yc = min(max(y0, 0), s.H - 1), xc = min(max(x0, 0), s.W - 1);
                        base = ((rr.bH + yc) * s.W + xc) * C;
                        base |= (tx0 && tx1) ? 1 : 0;
                        base |= (ty0 && ty1) ? 2 : 0;
                        w0 = (ty0 && tx0) ? w0 : 0.f;
                        w1 = (ty0 && tx1) ? w1 : 0.f;
                        w2 = (ty1 && tx0) ? w2 : 0.f;
                        w3 = (ty1 && tx1) ? w3 : 0.f;
                    }
                    const int e = g * TAB_STRIDE;
                    tb[e] = in ? base : 0;
                    tw[e] = in ? w0 : 0.f;
                    tw[e + tab_n] = in ? w1 : 0.f;
                    tw[e + 2 * tab_n] = in ? w2 : 0.f;
                    tw[e + 3 * tab_n] = in ? w3 : 0.f;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&tab_full[d_slot]);
            if (++d_tap == K) d_tap = 0;
        };
        // two raw sets in flight: the loads of table kb+2 are issued before table kb+1 is decoded
        RawRow ra, rb;
        ra.yx = rb.yx = -1;
        ra.bH = rb.bH = 0;
        ra.r.mi = rb.r.mi = 0;
        ra.r.fyx = rb.r.fyx = -1;
#pragma unroll
        for (int g = 0; g < GS; ++g) ra.r.dy[g] = ra.r.dx[g] = ra.r.mk[g] = rb.r.dy[g] = rb.r.dx[g] = rb.r.mk[g] = 0.f;
        if (total_kb > 0) {
            decode_rows(l_tile);
            load_next(ra, 0);
        }
        if (total_kb > 1) load_next(rb, 1);
        for (int kb = 0; kb < total_kb; kb += 2) {
            decode_store(ra, kb);
            if (kb + 2 < total_kb) load_next(ra, kb + 2);
            if (kb + 1 < total_kb) {
                decode_store(rb, kb + 1);
                if (kb + 3 < total_kb) load_next(rb, kb + 3);
            }
        }
    } else {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) dcn_mma_issuer<X3>(prm, smem, full, empty, tfull, tempty, tmem_base, nkb_tile);
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == S_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

int dcn_pack_weights(const float* w, float* wt, int Co, int C, int K, cudaStream_t st, bool x3) {
    if (x3) {
        MREFSR_CHECK(C % TBK_X3 == 0, ERR_BAD_ARG, "pack_weights (x3): C %% 16 != 0 (C = %d)", C);
        dcn_weight_repack_x3_kernel<<<cdiv(Co * C * K, 256), 256, 0, st>>>(w, wt, Co, C, K);
    } else {
        dcn_weight_repack_kernel<<<cdiv(Co * C * K, 256), 256, 0, st>>>(w, wt, Co, C, K);
    }
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

int dcn_nchw_to_nhwc(const float* x, float* xt, int B, int C, int HW, cudaStream_t st, bool round_tf32, float* xt_lo) {
    const dim3 grid(cdiv(HW, 32), cdiv(C, 128), B);
    if (xt_lo) nchw_to_nhwc_kernel<true, true><<<grid, 256, 0, st>>>(x, xt, C, HW, xt_lo);
    else if (round_tf32) nchw_to_nhwc_kernel<true><<<grid, 256, 0, st>>>(x, xt, C, HW, nullptr);
    else nchw_to_nhwc_kernel<false><<<grid, 256, 0, st>>>(x, xt, C, HW, nullptr);
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
bool dcn_tc_eligible(const DcnShape& s) {
    const int cdg = s.C / s.DG;
    // a 32-channel slab must cover whole deform groups (cdg | 32) or lie inside one (32 | cdg)
    const bool slab_ok = (cdg >= TBK) ? (cdg % TBK == 0) : (TBK % cdg == 0 && cdg % 8 == 0);
    return s.G == 1 && s.C % TBK == 0 && slab_ok && s.Co % 32 == 0 && s.Co >= 32 && s.Co <= 256 &&
           (size_t)s.B * s.C * s.H * s.W < ((size_t)1 << 31) && s.Ho < 32768 && s.Wo < 65536;
}

size_t dcn_tc_workspace_bytes(const DcnShape& s, int mode) {
    if (mode == MREFSR_DCN_FP32 || !dcn_tc_eligible(s)) return 0;
    const size_t wfloats = (size_t)s.Co * s.C * s.kh * s.kw * (mode == MREFSR_DCN_TF32X3 ? 2 : 1);   // X3: hi + lo
    return align_up((size_t)s.B * s.C * s.H * s.W * 4, 1024) + align_up(wfloats * 4, 1024);
}

// Row -> position mapping of the CTA tiles for prm.s (fills tiles, tile2d and the patch geometry)
static void dcn_plan_tiles(DcnTcParams& prm) {
    const DcnShape& s = prm.s;
    prm.tiles = cdiv(prm.total_rows, TBM);
    prm.tile2d = prm.tx_log = prm.ty_log = prm.sub_log = prm.subs_log = prm.nsx = prm.nsub = 0;
    // patch shape with the fewest padding rows; near-ties go to the larger patch (more neighbours share corners)
    static const int cand[5][2] = {{4, 4}, {4, 3}, {3, 4}, {3, 3}, {5, 3}};   // log2 (x, y): 16x16, 16x8, 8x16, 8x8, 32x8
    long long best = -1;
    for (int k = 0; k < 5; ++k) {
        const int tx = cand[k][0], ty = cand[k][1];
        const long long nsx = cdiv(s.Wo, 1 << tx), nsy = cdiv(s.Ho, 1 << ty);
        const long long rows = (long long)s.B * nsx * nsy << (tx + ty);
        const long long tiles = (rows + TBM - 1) / TBM;
        if (best < 0 || tiles * 100 < best * 97) {
            best = tiles;
            prm.tx_log = tx;
            prm.ty_log = ty;
            prm.nsx = (int)nsx;
            prm.nsub = (int)(nsx * nsy);
        }
    }
    // patches pay ~3-10 % (measured, profiles/r01s_dcn_ab.md); feature grids that tile badly (75 x 75: +14 % rows)
    // stay on the linear mapping
    if (best * 100 <= (long long)prm.tiles * 103) {
        prm.tile2d = 1;
        prm.sub_log = prm.tx_log + prm.ty_log;
        prm.subs_log = 8 - prm.sub_log;        // TBM = 256 rows = 2^subs_log patches
        prm.tiles = (int)best;
    }
}

// Test hook (host only, no device work): the tile plan of a [B, *, Ho, Wo] output and, when `coords` is given, the
// (sample, oy, ox) of every row of every tile (-1, -1, -1 for padding rows).  meta = {tile2d, patch_w, patch_h, tiles}.
int dcn_tc_tile_plan(int B, int Ho, int Wo, int* meta, int* coords, size_t max_rows) {
    DcnTcParams prm;
    memset(&prm, 0, sizeof(prm));
    prm.s.B = B;
    prm.s.Ho = Ho;
    prm.s.Wo = Wo;
    prm.P = Ho * Wo;
    prm.total_rows = B * prm.P;
    dcn_plan_tiles(prm);
    meta[0] = prm.tile2d;
    meta[1] = prm.tile2d ? 1 << prm.tx_log : TBM;
    meta[2] = prm.tile2d ? 1 << prm.ty_log : 1;
    meta[3] = prm.tiles;
    if (coords) {
        MREFSR_CHECK((size_t)prm.tiles * TBM <= max_rows, ERR_BAD_ARG, "tile plan: %d rows, room for %zu", prm.tiles * TBM,
                     max_rows);
        for (int t = 0; t < prm.tiles; ++t)
            for (int r = 0; r < TBM; ++r) {
                int b = -1, oy = -1, ox = -1;
                if (!dcn_row_coords(prm, t, r, b, oy, ox)) b = oy = ox = -1;
                int* c = coords + ((size_t)t * TBM + r) * 3;
                c[0] = b;
                c[1] = oy;
                c[2] = ox;
            }
    }
    return 0;
}

static int make_weight_map(CUtensorMap* map, const float* wt, int Co, int Ktot) {
    // 2-D tensor [Co rows][Ktot cols] fp32, box = 32 cols x Co rows, 128-byte swizzle; encoded as 3-D with d2 = 1
    return make_tensor_map_3d(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, wt, (uint64_t)Ktot, (uint64_t)Co, 1, TBK,
                              (uint32_t)Co, CU_TENSOR_MAP_SWIZZLE_128B);
}

int dcn_forward_tc_impl(const float* x, const float* w, const float* bias, const float* off, const float* mask,
                        const long long* max_idx, int flow_scale, float* out, const DcnShape& s, void* workspace,
                        size_t workspace_bytes, cudaStream_t st, int layout_flags, float out_slope,
                        const DcnOutputs* multi) {
    const bool x3 = (layout_flags & MREFSR_DCN_X3) != 0;
    const size_t need = dcn_tc_workspace_bytes(s, x3 ? MREFSR_DCN_TF32X3 : MREFSR_DCN_TF32);
    MREFSR_CHECK(workspace && workspace_bytes >= need, ERR_WORKSPACE, "dcn forward: workspace too small (%zu < %zu)",
                 workspace_bytes, need);
    MREFSR_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, ERR_WORKSPACE,
                 "dcn forward: workspace must be 1024-byte aligned");
    float* xt = static_cast<float*>(workspace);
    float* wt = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + align_up((size_t)s.B * s.C * s.H * s.W * 4, 1024));
    const int K = s.kh * s.kw, HW = s.H * s.W;
    {
        ScopedTiming tm(MREFSR_K_DCN_AUX, st);
        if (layout_flags & MREFSR_DCN_IN_NHWC) {      // the caller's tensor already is the gather layout
            MREFSR_CHECK((reinterpret_cast<uintptr_t>(x) & 31) == 0, ERR_BAD_ARG, "dcn forward: NHWC input must be 32-byte aligned");
            xt = const_cast<float*>(x);
        } else {
            nchw_to_nhwc_kernel<false><<<dim3(cdiv(HW, 32), cdiv(s.C, 128), s.B), 256, 0, st>>>(x, xt, s.C, HW, nullptr);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        }
        if (layout_flags & MREFSR_DCN_W_PACKED) {      // packed once by the caller (mrefsr_dcn_pack_weights[_x3])
            MREFSR_CHECK((reinterpret_cast<uintptr_t>(w) & 15) == 0, ERR_BAD_ARG, "dcn forward: packed weights must be 16-byte aligned");
            wt = const_cast<float*>(w);
        } else {
            int prc = dcn_pack_weights(w, wt, s.Co, s.C, K, st, x3);
            if (prc) return prc;
        }
    }
    CUtensorMap mapW;
    int rc = make_weight_map(&mapW, wt, s.Co, K * s.C * (x3 ? 2 : 1));
    if (rc) return rc;
    DcnTcParams prm;
    prm.s = s;
    prm.P = s.Ho * s.Wo;
    prm.total_rows = s.B * prm.P;
    dcn_plan_tiles(prm);
    const int slab = x3 ? TBK_X3 : TBK;     // channels per K step (every eligible shape has C % 32 == 0, cdg % 8 == 0)
    prm.n_slabs = s.C / slab;
    prm.taps = K;
    prm.cdg = s.C / s.DG;
    prm.gs = prm.cdg >= slab ? 1 : slab / prm.cdg;
    prm.stage_bytes = T_A_BYTES + s.Co * 128;
    const size_t table_bytes = (size_t)S_NTAB * 5 * prm.gs * (TBM + 4) * 4;
    // stage ring vs L1: at 8 channels per deform group the gather needs the L1 more than a third stage (2.11 vs 1.91 ms
    // at the large scale); from 16 channels per group on, the third stage wins now that the gather groups alternate
    int smem_budget = prm.cdg >= 16 ? 205 * 1024 : T_SMEM_BUDGET;
#ifdef MREFSR_DCN_DEBUG
    if (getenv("MREFSR_DCN_SMEM_KB")) smem_budget = atoi(getenv("MREFSR_DCN_SMEM_KB")) * 1024;   // tuning experiments
#endif
    prm.stages = (int)((smem_budget - (int)table_bytes) / prm.stage_bytes);
    if (prm.stages > 4) prm.stages = 4;
    if (prm.stages < 2) prm.stages = 2;
    prm.nbuf = (2 * s.Co * 2 <= 512) ? 2 : 1;
    prm.fused = max_idx != nullptr;
    prm.dbg = 0;
#ifdef MREFSR_DCN_DEBUG
    prm.dbg = getenv("MREFSR_DCN_DBG") ? atoi(getenv("MREFSR_DCN_DBG")) : 0;
#endif
    for (int k = 0; k < 8; ++k) prm.outs[k] = nullptr;
    if (multi) {
        MREFSR_CHECK(multi->n >= 1 && multi->n <= 8, ERR_BAD_ARG, "dcn forward: 1..8 output buffers (got %d)", multi->n);
        MREFSR_CHECK(multi->group >= 0 && (multi->group == 0 || s.B % multi->group == 0), ERR_BAD_ARG,
                     "dcn forward: batch %d not a multiple of the destination group %d", s.B, multi->group);
        for (int k = 0; k < multi->n; ++k) {
            MREFSR_CHECK(multi->ptr[k], ERR_BAD_ARG, "dcn forward: output buffer %d is NULL", k);
            prm.outs[k] = multi->ptr[k];
        }
        prm.n_outs = multi->n;
        prm.dst_group = multi->group;
        prm.dst_stride = multi->stride;
        prm.dst_offset = multi->offset;
        prm.dst_slab_rows = multi->slab_rows;
        MREFSR_CHECK(multi->slab_rows >= 0 && (multi->slab_rows == 0 || (!(layout_flags & MREFSR_DCN_OUT_NHWC) &&
                     (long long)multi->slab_rows * multi->n >= s.Ho)), ERR_BAD_ARG,
                     "dcn forward: slab routing needs NCHW outputs and slab_rows * buffers >= output rows");
    } else {
        prm.outs[0] = out;
        prm.n_outs = 1;
        prm.dst_group = prm.dst_stride = prm.dst_offset = prm.dst_slab_rows = 0;
    }
    prm.out_nhwc = (layout_flags & MREFSR_DCN_OUT_NHWC) ? 1 : 0;
    prm.out_slope = out_slope;

    prm.flow_scale = flow_scale;
    prm.hp = prm.wp = 0;
    prm.wp_magic = 0;
    if (prm.fused) {
        MREFSR_CHECK(flow_scale >= 1 && s.Ho % flow_scale == 0 && s.Wo % flow_scale == 0, ERR_BAD_ARG,
                     "fused DynAgg: output %dx%d not a multiple of the flow scale %d", s.Ho, s.Wo, flow_scale);
        prm.hp = s.Ho / flow_scale - 2;
        prm.wp = s.Wo / flow_scale - 2;
        MREFSR_CHECK(prm.hp > 0 && prm.wp > 1, ERR_BAD_ARG, "fused DynAgg: feature grid too small");
        MREFSR_CHECK((unsigned long long)prm.hp * prm.wp * prm.wp < (1ull << 32), ERR_BAD_ARG,
                     "fused DynAgg: feature grid %dx%d too large", prm.hp, prm.wp);
        prm.wp_magic = 0xFFFFFFFFu / (unsigned)prm.wp + 1u;
    }
    const size_t smem = (size_t)prm.stages * prm.stage_bytes + 256 + table_bytes + 1024;
    int grid = sm_count();
    if (grid > prm.tiles) grid = prm.tiles;
    using Kernel = decltype(&dcn_tc_split_kernel<false, 1>);
    static const Kernel kernels[2][3] = {   // [FUSED][GS = 1, 2, 4]
        {dcn_tc_split_kernel<false, 1>, dcn_tc_split_kernel<false, 2>, dcn_tc_split_kernel<false, 4>},
        {dcn_tc_split_kernel<true, 1>, dcn_tc_split_kernel<true, 2>, dcn_tc_split_kernel<true, 4>}};
    static const Kernel kernels_x3[2][2] = {   // [FUSED][GS = 1, 2]: 16-channel slabs hold at most two deform groups
        {dcn_tc_split_kernel<false, 1, true>, dcn_tc_split_kernel<false, 2, true>},
        {dcn_tc_split_kernel<true, 1, true>, dcn_tc_split_kernel<true, 2, true>}};
    const Kernel kern = x3 ? kernels_x3[prm.fused][prm.gs >> 1] : kernels[prm.fused][prm.gs >> 1];
    ScopedTiming tm(MREFSR_K_DCN_FWD, st);
    MREFSR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, S_THREADS, smem, st>>>(mapW, xt, off, prm.fused ? nullptr : mask, prm.fused ? max_idx : nullptr, bias,
                                        prm);
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

int dcn_forward_tc(const float* x, const float* w, const float* bias, const float* off, const float* mask, float* out,
                   const DcnShape& s, void* workspace, size_t workspace_bytes, cudaStream_t st, bool x3) {
    return dcn_forward_tc_impl(x, w, bias, off, mask, nullptr, 1, out, s, workspace, workspace_bytes, st,
                               x3 ? MREFSR_DCN_X3 : 0, 1.f, nullptr);
}

}  // namespace mrefsr
