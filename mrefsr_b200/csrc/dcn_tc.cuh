// mrefsr_b200/csrc/dcn_tc.cuh -- the tcgen05 DCN forward's tile geometry, parameters and device helpers
// (dcn_tc.cu); dcn.cu's backward shares the tf32 rounding.
#pragma once
#include "dcn_common.cuh"

namespace mrefsr {

constexpr int TBM = 256;            // rows (output positions) per CTA tile
constexpr int TBK = 32;             // fp32 channels per K step (128-byte rows)
constexpr int TBK_X3 = 16;          // channels per K step of the 3-pass kernels: a 128-byte row is [hi 16 | lo 16]
constexpr int T_A_BYTES = TBM * 128;
constexpr int T_SMEM_BUDGET = 150 * 1024;          // stage ring; the rest of the 228 KB stays L1 for the gather

struct DcnTcParams {
    DcnShape s;
    int P, total_rows, tiles, n_slabs, taps, cdg, gs, stages, nbuf, stage_bytes;
    // fused DynAgg mode
    int fused, flow_scale, hp, wp;
    // Outputs: the epilogue stores every finished tile to each of n_outs buffers (this GPU's and, in the
    // reference-sharded mode, the peers' copies of the gathered tensor, mapped over NVLink), at sample slot
    // (b / dst_group) * dst_stride + dst_offset + b % dst_group  (dst_group == 0: slot b).
    float* outs[8];
    int n_outs, dst_group, dst_stride, dst_offset;
    // dst_slab_rows > 0 (NCHW outputs only): pixel-slab routing -- output row oy belongs to buffer oy / dst_slab_rows
    // ALONE, which holds [slots, Co, dst_slab_rows, Wo]: each rank of the reference-sharded mode then receives only
    // the rows it fuses (an all-to-all folded into the epilogue instead of an all-gather)
    int dst_slab_rows;
    int out_nhwc;        // epilogue writes [B, Ho, Wo, Co] instead of [B, Co, Ho, Wo]
    float out_slope;     // leaky-ReLU slope applied to the output (1: none)
    unsigned wp_magic;   // ceil(2^32 / wp): idx / wp == umulhi(idx, wp_magic) for idx < hp * wp  (hp * wp * wp < 2^32)
    // Row -> output position mapping of a CTA tile.  tile2d == 0: rows are 256 consecutive positions of the
    // B*Ho*Wo concatenation.  tile2d == 1: the tile is 2^subs_log square-ish patches of 2^tx_log x 2^ty_log
    // positions (nsx patches per output row, nsub per sample), so that the bilinear corners of x- AND y-neighbours
    // fall into the same K step and hit in L1.
    int tile2d, tx_log, ty_log, sub_log, subs_log, nsx, nsub;
    int dbg;             // ablation bits, read by variant builds only (MREFSR_DCN_DEBUG)
};

// (tile, row within the tile) -> (sample, oy, ox); false for padding rows
__host__ __device__ __forceinline__ bool dcn_row_coords(const DcnTcParams& prm, int tile, int r, int& b, int& oy, int& ox) {
    if (!prm.tile2d) {
        const int m = tile * TBM + r;
        if (m >= prm.total_rows) return false;
        b = m / prm.P;
        const int p = m - b * prm.P;
        oy = p / prm.s.Wo;
        ox = p - oy * prm.s.Wo;
        return true;
    }
    const int st = (tile << prm.subs_log) + (r >> prm.sub_log);   // patch index over the whole batch
    const int within = r & ((1 << prm.sub_log) - 1);
    b = st / prm.nsub;
    const int rem = st - b * prm.nsub, ty = rem / prm.nsx, tx = rem - ty * prm.nsx;
    oy = (ty << prm.ty_log) + (within >> prm.tx_log);
    ox = (tx << prm.tx_log) + (within & ((1 << prm.tx_log) - 1));
    return b < prm.s.B && oy < prm.s.Ho && ox < prm.s.Wo;
}

__device__ __forceinline__ float to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// Loads whose issue point matters (software pipelining): volatile asm keeps program order with respect to the
// mbarrier waits, so the compiler cannot sink them down to their first use one K step later.
__device__ __forceinline__ float ldg_early(const float* p) {
    float v;
    // offsets / masks are read exactly once: keep them out of L1, which the gather needs
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ long long ldg_early_s64(const long long* p) {
    long long v;
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}

// round-to-nearest (ties away) to tf32 in one integer add: the tensor core ignores the low 13 mantissa bits
__device__ __forceinline__ float tf32_round_bits(float v) { return __uint_as_float(__float_as_uint(v) + 0x1000u); }

// 3-pass split of v: hi = v rounded to tf32 with the low bits CLEARED (v - hi must be the exact remainder, so hi cannot
// rely on the tensor core's truncation), lo = the remainder rounded like tf32_round_bits.  hi + lo carries 22 bits.
__device__ __forceinline__ void tf32_split_bits(float v, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & ~0x1FFFu);
    lo = tf32_round_bits(v - hi);
}

// 256-bit read-only load: 8 consecutive channels of one corner (one full 32-byte sector per lane)
struct F8 {
    float2 v[4];
};
__device__ __forceinline__ F8 ldg8(const float* p) {
    F8 r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(r.v[0].x), "=f"(r.v[0].y), "=f"(r.v[1].x), "=f"(r.v[1].y), "=f"(r.v[2].x), "=f"(r.v[2].y),
          "=f"(r.v[3].x), "=f"(r.v[3].y)
        : "l"(p));
    return r;
}
constexpr int TAB_STRIDE = TBM + 4;   // per-group row stride of the sample table (+4: no bank conflicts)

__device__ __forceinline__ int ldg_early_s32(const int* p) {
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

}  // namespace mrefsr
