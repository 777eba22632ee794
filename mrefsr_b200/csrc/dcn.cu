// mrefsr_b200/csrc/dcn.cu -- modulated deformable convolution (DCNv2): exact-fp32 CUDA-core forward, backward,
// and the DynAgg offset/mask glue.  The tcgen05 (TF32) forward lives in dcn_tc.cu.
//
// Replaces basicsr/ops/dcn/src/deform_conv_cuda.cpp:490-685 and the kernels of
// basicsr/ops/dcn/src/deform_conv_cuda_kernel.cu:468-767.  Differences in structure (not in results):
//   * forward: no columns buffer and no per-sample loop -- the bilinear gather feeds the GEMM tile directly
//     from shared memory, batched over B in one launch (the reference launches im2col + addmm_ per sample,
//     deform_conv_cuda.cpp:539-555);
//   * backward: the reference's per-sample {addmm_, col2im_coord, col2im, im2col, addmm_ x2} sequence
//     (deform_conv_cuda.cpp:612-672) is batched over chunks of samples sized to a bounded workspace.
#include <type_traits>

#include "common.cuh"
#include "dcn_tc.cuh"
#include "../../include/mrefsr_b200.h"

namespace mrefsr {

constexpr int DT = 64;  // tile edge of the CUDA-core GEMM tiles
constexpr int DK = 16;  // K step

// =====================================================================================================
// forward, exact fp32: tile = 64 output positions x 64 output channels, K = (tap, 16 input channels)
// grid (ceil(P/64), G * ceil(Co/G/64), B), block 256
// =====================================================================================================
__global__ void __launch_bounds__(256)
dcn_fwd_simt_kernel(const float* __restrict__ x, const float* __restrict__ offset, const float* __restrict__ mask,
                    const float* __restrict__ weight, const float* __restrict__ bias, float* __restrict__ out,
                    const DcnShape s) {
    __shared__ float As[DK][DT + 4];
    __shared__ float Bs[DK][DT + 4];
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cpg = s.C / s.G, opg = s.Co / s.G, cdg = s.C / s.DG;
    const int oct = cdiv_d(opg, DT);
    const int b = blockIdx.z, gi = blockIdx.y / oct, ot = blockIdx.y % oct;
    const int p0 = blockIdx.x * DT, oc0 = ot * DT;  // oc0 is group-local
    const int t = threadIdx.x;
    const int lpos = t & 63, lkq = (t >> 6) * 4;
    const int ty = t >> 4, tx = t & 15;
    const int p = p0 + lpos;
    const bool pvalid = p < P;
    const int oy = pvalid ? p / s.Wo : 0, ox = pvalid ? p % s.Wo : 0;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int tap = 0; tap < K; ++tap) {
        const int ti = tap / s.kw, tj = tap % s.kw;
        const float ybase = (float)(oy * s.sh - s.ph + ti * s.dh), xbase = (float)(ox * s.sw - s.pw + tj * s.dw);
        for (int c0 = 0; c0 < cpg; c0 += DK) {
            // ---- A tile: gathered, modulated samples
            int last_dg = -1;
            float sy = 0.f, sx = 0.f, sm = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int cl = c0 + lkq + e;
                float v = 0.f;
                if (pvalid && cl < cpg) {
                    const int ch = gi * cpg + cl;
                    const int dgi = ch / cdg;
                    if (dgi != last_dg) {
                        const size_t ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
                        sy = ybase + __ldg(offset + ob);
                        sx = xbase + __ldg(offset + ob + P);
                        sm = mask ? __ldg(mask + ((size_t)(b * s.DG + dgi) * K + tap) * P + p) : 1.f;
                        last_dg = dgi;
                    }
                    v = dcn_sample(x + ((size_t)b * s.C + ch) * s.H * s.W, s.H, s.W, sy, sx) * sm;
                }
                As[lkq + e][lpos] = v;
            }
            // ---- B tile: weights W[oc][c][tap]
            {
                const int oc = oc0 + lpos;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int cl = c0 + lkq + e;
                    float v = 0.f;
                    if (oc < opg && cl < cpg) v = __ldg(weight + ((size_t)(gi * opg + oc) * cpg + cl) * K + tap);
                    Bs[lkq + e][lpos] = v;
                }
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < DK; ++k) {
                const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
                const float4 bb = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
                const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ocl = oc0 + tx * 4 + j;
        if (ocl >= opg) continue;
        const int oc = gi * opg + ocl;
        const float bv = bias ? __ldg(bias + oc) : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int pp = p0 + ty * 4 + i;
            if (pp < P) out[((size_t)b * s.Co + oc) * P + pp] = acc[i][j] + bv;
        }
    }
}

// =====================================================================================================
// backward
// =====================================================================================================
template <class Src>
constexpr bool kDynAgg = std::is_same<Src, DynAggSrc>::value;

// Sampling point (y, x) and mask m of (sample b, deform group dgi, tap, output position) from the DynAgg-fused source,
// bit for bit as the fused forward's decode warps compute them (dcn_tc.cu, load_next / decode_store): the flow of
// max_idx[b][oy/s - i][ox/s - j] (0 outside the hp x wp grid) added to the learned offset first, then the tap's base
// position, and the fast-intrinsic sigmoid.  Forward and backward must sample the same points: the offset gradient
// jumps at cell edges.  Returns the index of the dy plane element in conv_out (dx: + P); *mc = that of the mask logit.
__device__ __forceinline__ size_t dynagg_point(const float* __restrict__ conv_out, const DynAggSrc& f, const DcnShape& s,
                                               int b, int dgi, int tap, int oy, int ox, float& y, float& x, float& m,
                                               size_t& mc) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, ti = tap / s.kw, tj = tap - ti * s.kw;
    const size_t base = (size_t)b * 3 * s.DG * K * P + (size_t)oy * s.Wo + ox;
    const size_t oc = base + (size_t)2 * (dgi * K + tap) * P;
    mc = base + (size_t)(2 * s.DG * K + dgi * K + tap) * P;
    float fly = 0.f, flx = 0.f;
    const int fy = oy / f.flow_scale - ti, fx = ox / f.flow_scale - tj;
    if (fy >= 0 && fx >= 0 && fy < f.hp && fx < f.wp) {
        const int mi = (int)__ldg(f.max_idx + ((size_t)b * f.hp + fy) * f.wp + fx);
        const int my = mi / f.wp, mx = mi - my * f.wp;
        fly = (float)((my - fy) * f.flow_scale);
        flx = (float)((mx - fx) * f.flow_scale);
    }
    y = (float)(oy * s.sh - s.ph + ti * s.dh) + (__ldg(conv_out + oc) + fly);
    x = (float)(ox * s.sw - s.pw + tj * s.dw) + (__ldg(conv_out + oc + P) + flx);
    m = __fdividef(1.f, 1.f + __expf(-__ldg(conv_out + mc)));
    return oc;
}

__host__ __device__ __forceinline__ bool src_nhwc(const PlaneSrc&) { return false; }
__host__ __device__ __forceinline__ bool src_nhwc(const DynAggSrc& f) { return f.x_nhwc != 0; }

// dcn_sample on channel `ch` of sample `xb` in either input layout (NHWC: pixels C floats apart)
__device__ __forceinline__ float dcn_sample_any(const float* __restrict__ xb, int ch, const DcnShape& s, bool nhwc, float y,
                                                float x) {
    if (!nhwc) return dcn_sample(xb + (size_t)ch * s.H * s.W, s.H, s.W, y, x);
    if (!(y > -1.f && x > -1.f && y < (float)s.H && x < (float)s.W)) return 0.f;
    const float* pl = xb + ch;
    const int y0 = (int)floorf(y), x0 = (int)floorf(x);
    const int y1 = y0 + 1, x1 = x0 + 1;
    const float ly = y - (float)y0, lx = x - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const float a = (y0 >= 0 && x0 >= 0) ? __ldg(pl + (y0 * s.W + x0) * s.C) : 0.f;
    const float b = (y0 >= 0 && x1 <= s.W - 1) ? __ldg(pl + (y0 * s.W + x1) * s.C) : 0.f;
    const float c = (y1 <= s.H - 1 && x0 >= 0) ? __ldg(pl + (y1 * s.W + x0) * s.C) : 0.f;
    const float d = (y1 <= s.H - 1 && x1 <= s.W - 1) ? __ldg(pl + (y1 * s.W + x1) * s.C) : 0.f;
    return hy * hx * a + hy * lx * b + ly * hx * c + ly * lx * d;
}

// (1) gcol[bl][(ch*K+tap)][p] = sum_oc W[oc][(c*K+tap)] * gout[b][oc][p]     (deform_conv_cuda.cpp:623-626)
// grid (ceil(P/64), G * ceil(cpg*K/64), nb), block 256
__global__ void __launch_bounds__(256)
dcn_bwd_gcol_kernel(const float* __restrict__ weight, const float* __restrict__ gout, float* __restrict__ gcol,
                    const DcnShape s, int b0) {
    __shared__ float As[DK][DT + 4];
    __shared__ float Bs[DK][DT + 4];
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cpg = s.C / s.G, opg = s.Co / s.G, MK = cpg * K;
    const int mt_per = cdiv_d(MK, DT);
    const int bl = blockIdx.z, b = b0 + bl, gi = blockIdx.y / mt_per, mt = blockIdx.y % mt_per;
    const int p0 = blockIdx.x * DT, m0 = mt * DT;
    const int t = threadIdx.x, lidx = t & 63, lkq = (t >> 6) * 4, ty = t >> 4, tx = t & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < opg; k0 += DK) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = k0 + lkq + e;
            const int m = m0 + lidx, pp = p0 + lidx;
            As[lkq + e][lidx] = (k < opg && m < MK) ? __ldg(weight + (size_t)(gi * opg + k) * MK + m) : 0.f;
            Bs[lkq + e][lidx] = (k < opg && pp < P) ? __ldg(gout + ((size_t)b * s.Co + gi * opg + k) * P + pp) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < DK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 bb = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= MK) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int pp = p0 + tx * 4 + j;
            if (pp < P) gcol[((size_t)bl * s.C * K + (size_t)gi * MK + m) * P + pp] = acc[i][j];
        }
    }
}

// (2) grad_offset / grad_mask  (.cu:695-767): one thread per (bl, deform group, tap, position)
__global__ void dcn_bwd_coord_kernel(const float* __restrict__ x, const float* __restrict__ offset,
                                     const float* __restrict__ mask, const float* __restrict__ gcol,
                                     float* __restrict__ goff, float* __restrict__ gmask, const DcnShape s, int b0,
                                     int nb) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.DG * K * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int tap = (idx / P) % K;
        const int dgi = (idx / ((size_t)P * K)) % s.DG;
        const int bl = idx / ((size_t)P * K * s.DG);
        const int b = b0 + bl;
        const int oy = p / s.Wo, ox = p % s.Wo, ti = tap / s.kw, tj = tap % s.kw;
        const size_t ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
        const size_t mb = ((size_t)(b * s.DG + dgi) * K + tap) * P + p;
        const float y = (float)(oy * s.sh - s.ph + ti * s.dh) + offset[ob];
        const float xx = (float)(ox * s.sw - s.pw + tj * s.dw) + offset[ob + P];
        const float m = mask ? mask[mb] : 1.f;
        float dy = 0.f, dx = 0.f, dm = 0.f;
        if (y > -1.f && xx > -1.f && y < (float)s.H && xx < (float)s.W) {
            const int y0 = (int)floorf(y), x0 = (int)floorf(xx), y1 = y0 + 1, x1 = x0 + 1;
            const float ly = y - y0, lx = xx - x0;
            const bool va = y0 >= 0 && x0 >= 0, vb = y0 >= 0 && x1 <= s.W - 1, vc = y1 <= s.H - 1 && x0 >= 0,
                       vd = y1 <= s.H - 1 && x1 <= s.W - 1;
            for (int cc = 0; cc < cdg; ++cc) {
                const int ch = dgi * cdg + cc;
                const float* pl = x + ((size_t)b * s.C + ch) * s.H * s.W;
                const float a = va ? __ldg(pl + y0 * s.W + x0) : 0.f;
                const float bq = vb ? __ldg(pl + y0 * s.W + x1) : 0.f;
                const float cq = vc ? __ldg(pl + y1 * s.W + x0) : 0.f;
                const float d = vd ? __ldg(pl + y1 * s.W + x1) : 0.f;
                const float gc = gcol[((size_t)bl * s.C * K + (size_t)ch * K + tap) * P + p];
                const float v = (1.f - ly) * (1.f - lx) * a + (1.f - ly) * lx * bq + ly * (1.f - lx) * cq + ly * lx * d;
                dm += gc * v;
                dy += gc * m * ((1.f - lx) * (cq - a) + lx * (d - bq));
                dx += gc * m * ((1.f - ly) * (bq - a) + ly * (d - cq));
            }
        }
        goff[ob] = dy;
        goff[ob + P] = dx;
        if (gmask) gmask[mb] = dm;
    }
}

// (3) grad_input: bilinear scatter of gcol * mask (.cu:635-693), one thread per (bl, channel, tap, position)
__global__ void dcn_bwd_input_kernel(const float* __restrict__ offset, const float* __restrict__ mask,
                                     const float* __restrict__ gcol, float* __restrict__ gx, const DcnShape s, int b0,
                                     int nb, const PlaneSrc) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.C * K * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int tap = (idx / P) % K;
        const int ch = (idx / ((size_t)P * K)) % s.C;
        const int bl = idx / ((size_t)P * K * s.C);
        const int b = b0 + bl, dgi = ch / cdg;
        const int oy = p / s.Wo, ox = p % s.Wo, ti = tap / s.kw, tj = tap % s.kw;
        const size_t ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
        const float y = (float)(oy * s.sh - s.ph + ti * s.dh) + offset[ob];
        const float xx = (float)(ox * s.sw - s.pw + tj * s.dw) + offset[ob + P];
        if (!(y > -1.f && xx > -1.f && y < (float)s.H && xx < (float)s.W)) continue;
        const float tval = gcol[idx] * (mask ? mask[((size_t)(b * s.DG + dgi) * K + tap) * P + p] : 1.f);
        const int y0 = (int)floorf(y), x0 = (int)floorf(xx), y1 = y0 + 1, x1 = x0 + 1;
        const float ly = y - y0, lx = xx - x0;
        float* pl = gx + ((size_t)b * s.C + ch) * s.H * s.W;
        if (y0 >= 0 && x0 >= 0) atomicAdd(pl + y0 * s.W + x0, (1.f - ly) * (1.f - lx) * tval);
        if (y0 >= 0 && x1 <= s.W - 1) atomicAdd(pl + y0 * s.W + x1, (1.f - ly) * lx * tval);
        if (y1 <= s.H - 1 && x0 >= 0) atomicAdd(pl + y1 * s.W + x0, ly * (1.f - lx) * tval);
        if (y1 <= s.H - 1 && x1 <= s.W - 1) atomicAdd(pl + y1 * s.W + x1, ly * lx * tval);
    }
}

// DynAggSrc: `offset` is conv_out, mask unused; grad_input in the input's layout (src.x_nhwc: [B, H, W, C])
__global__ void dcn_bwd_input_kernel(const float* __restrict__ offset, const float* __restrict__ mask,
                                     const float* __restrict__ gcol, float* __restrict__ gx, const DcnShape s, int b0,
                                     int nb, const DynAggSrc src) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.C * K * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int tap = (idx / P) % K;
        const int ch = (idx / ((size_t)P * K)) % s.C;
        const int bl = idx / ((size_t)P * K * s.C);
        const int b = b0 + bl, dgi = ch / cdg;
        const int oy = p / s.Wo, ox = p % s.Wo, ti = tap / s.kw, tj = tap % s.kw;
        float y, xx, m;
        size_t mc;
        dynagg_point(offset, src, s, b, dgi, tap, oy, ox, y, xx, m, mc);
        if (!(y > -1.f && xx > -1.f && y < (float)s.H && xx < (float)s.W)) continue;
        const float tval = gcol[idx] * m;
        const int y0 = (int)floorf(y), x0 = (int)floorf(xx), y1 = y0 + 1, x1 = x0 + 1;
        const float ly = y - y0, lx = xx - x0;
        const int ps = src.x_nhwc ? s.C : 1;     // pixel stride of grad_input's channel `ch`
        float* pl = gx + (src.x_nhwc ? (size_t)b * s.C * s.H * s.W + ch : ((size_t)b * s.C + ch) * s.H * s.W);
        if (y0 >= 0 && x0 >= 0) atomicAdd(pl + (y0 * s.W + x0) * ps, (1.f - ly) * (1.f - lx) * tval);
        if (y0 >= 0 && x1 <= s.W - 1) atomicAdd(pl + (y0 * s.W + x1) * ps, (1.f - ly) * lx * tval);
        if (y1 <= s.H - 1 && x0 >= 0) atomicAdd(pl + (y1 * s.W + x0) * ps, ly * (1.f - lx) * tval);
        if (y1 <= s.H - 1 && x1 <= s.W - 1) atomicAdd(pl + (y1 * s.W + x1) * ps, ly * lx * tval);
    }
}

// (4a) columns[bl][(ch*K+tap)][p]  (.cu:571-633), recomputed for grad_weight like deform_conv_cuda.cpp:647-650
template <class Src>
__device__ __forceinline__ void dcn_im2col(const float* __restrict__ x, const float* __restrict__ offset,
                                  const float* __restrict__ mask, float* __restrict__ col, const DcnShape s, int b0,
                                  int nb, const Src& src) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.C * K * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int tap = (idx / P) % K;
        const int ch = (idx / ((size_t)P * K)) % s.C;
        const int bl = idx / ((size_t)P * K * s.C);
        const int b = b0 + bl, dgi = ch / cdg;
        const int oy = p / s.Wo, ox = p % s.Wo, ti = tap / s.kw, tj = tap % s.kw;
        if constexpr (kDynAgg<Src>) {
            float y, xx, m;
            size_t mc;
            dynagg_point(offset, src, s, b, dgi, tap, oy, ox, y, xx, m, mc);
            col[idx] = dcn_sample_any(x + (size_t)b * s.C * s.H * s.W, ch, s, src.x_nhwc, y, xx) * m;
            continue;
        }
        const size_t ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
        const float y = (float)(oy * s.sh - s.ph + ti * s.dh) + offset[ob];
        const float xx = (float)(ox * s.sw - s.pw + tj * s.dw) + offset[ob + P];
        const float m = mask ? mask[((size_t)(b * s.DG + dgi) * K + tap) * P + p] : 1.f;
        col[idx] = dcn_sample(x + ((size_t)b * s.C + ch) * s.H * s.W, s.H, s.W, y, xx) * m;
    }
}

// one kernel per sample source under one name (the source is the type of the last argument)
__global__ void dcn_im2col_kernel(const float* __restrict__ x, const float* __restrict__ offset, const float* __restrict__ mask,
                                  float* __restrict__ col, const DcnShape s, int b0, int nb, const PlaneSrc src) {
    dcn_im2col(x, offset, mask, col, s, b0, nb, src);
}
__global__ void dcn_im2col_kernel(const float* __restrict__ x, const float* __restrict__ offset, const float* __restrict__ mask,
                                  float* __restrict__ col, const DcnShape s, int b0, int nb, const DynAggSrc src) {
    dcn_im2col(x, offset, mask, col, s, b0, nb, src);
}

// (4a') columns from the NHWC copy of the input.  One thread = (position, tap, 8-channel chunk): one sample decode, four
// 256-bit corner loads; lanes = consecutive positions (coalesced offset / mask reads).  The planar kernel above issues
// 8x the L1 sectors.
struct __align__(32) Col8 {
    float v[8];
};
__device__ __forceinline__ Col8 ldg_col8(const float* p) {
    Col8 r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
        : "l"(p));
    return r;
}
// (2') grad_offset / grad_mask from the NHWC copy of the input: one thread per (bl, deform group, tap, position) like the
// planar kernel above, but the group's channels come as 8-channel chunks with four 256-bit corner loads each instead of
// 32 scalar plane loads per chunk.  One thread owns a whole (group, tap, position): plain stores, deterministic.
// DynAggSrc: goff is the gradient of the raw conv_offset_mask output (dy, dx and dm * m * (1 - m) at its channels).
template <class Src>
__device__ __forceinline__ void
dcn_bwd_coord_nhwc(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          const DcnShape s, int b0, int nb, const Src& src) {
    // thread = (bl, deform group, position), the taps are a loop: the nine sampling points of a position lie within a
    // few pixels of each other, so their corners meet in L1 (a thread per tap re-fetched every sector from L2 per tap)
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.DG * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int dgi = (idx / P) % s.DG;
        const int bl = idx / ((size_t)P * s.DG);
        const int b = b0 + bl;
        const int oy = p / s.Wo, ox = p - oy * s.Wo;
        const float* xb = xt + (size_t)b * s.H * s.W * s.C + dgi * cdg;
        for (int tap = 0; tap < K; ++tap) {
            const int ti = tap / s.kw, tj = tap - ti * s.kw;
            size_t ob, mb;
            float y, x, m;
            if constexpr (kDynAgg<Src>) {
                ob = dynagg_point(offset, src, s, b, dgi, tap, oy, ox, y, x, m, mb);
            } else {
                ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
                mb = ((size_t)(b * s.DG + dgi) * K + tap) * P + p;
                y = (float)(oy * s.sh - s.ph + ti * s.dh) + __ldcs(offset + ob);
                x = (float)(ox * s.sw - s.pw + tj * s.dw) + __ldcs(offset + ob + P);
                m = mask ? __ldcs(mask + mb) : 1.f;
            }
            float dy = 0.f, dx = 0.f, dm = 0.f;
            if (y > -1.f && x > -1.f && y < (float)s.H && x < (float)s.W) {
                const float fy0 = floorf(y), fx0 = floorf(x);
                const int y0 = (int)fy0, x0 = (int)fx0;
                const float ly = y - fy0, lx = x - fx0, hy = 1.f - ly, hx = 1.f - lx;
                const bool ty0 = y0 >= 0, ty1 = y0 + 1 <= s.H - 1, tx0 = x0 >= 0, tx1 = x0 + 1 <= s.W - 1;
                const int yc = ty0 ? y0 : 0, xc = tx0 ? x0 : 0;
                const float* base = xb + ((size_t)yc * s.W + xc) * s.C;
                const size_t dxo = (tx0 && tx1) ? s.C : 0, dyo = (ty0 && ty1) ? (size_t)s.W * s.C : 0;
                const float va = (ty0 && tx0) ? 1.f : 0.f, vb = (ty0 && tx1) ? 1.f : 0.f, vc = (ty1 && tx0) ? 1.f : 0.f,
                            vd = (ty1 && tx1) ? 1.f : 0.f;
                const float* gc = gcol + ((size_t)bl * s.C * K + (size_t)dgi * cdg * K + tap) * P + p;
                for (int c0 = 0; c0 < cdg; c0 += 8) {
                    const Col8 v0 = ldg_col8(base + c0), v1 = ldg_col8(base + c0 + dxo), v2 = ldg_col8(base + c0 + dyo),
                               v3 = ldg_col8(base + c0 + dyo + dxo);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float a = va * v0.v[e], bq = vb * v1.v[e], cq = vc * v2.v[e], d = vd * v3.v[e];
                        const float g = __ldcs(gc + (size_t)(c0 + e) * K * P);      // read once: keep it out of the corners' L1
                        const float v = hy * hx * a + hy * lx * bq + ly * hx * cq + ly * lx * d;
                        dm += g * v;
                        dy += g * m * (hx * (cq - a) + lx * (d - bq));
                        dx += g * m * (hy * (bq - a) + ly * (d - cq));
                    }
                }
            }
            __stcs(goff + ob, dy);
            __stcs(goff + ob + P, dx);
            if constexpr (kDynAgg<Src>) __stcs(goff + mb, dm * m * (1.f - m));     // d sigmoid = m (1 - m)
            else if (gmask) __stcs(gmask + mb, dm);
        }
    }
}

__global__ void __launch_bounds__(256, 3)
dcn_bwd_coord_nhwc_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          const DcnShape s, int b0, int nb, const PlaneSrc src) {
    dcn_bwd_coord_nhwc(xt, offset, mask, gcol, goff, gmask, s, b0, nb, src);
}

__global__ void __launch_bounds__(256, 3)
dcn_bwd_coord_nhwc_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          const DcnShape s, int b0, int nb, const DynAggSrc src) {
    dcn_bwd_coord_nhwc(xt, offset, mask, gcol, goff, gmask, s, b0, nb, src);
}

// (2') + (4a') in one pass: the coordinate gradients and the recomputed columns need the same corners of the same sampling
// points, so when a backward wants both (grad_offset / grad_mask and grad_weight: every training step of MRefSR) one kernel
// gathers them once.  Thread = (bl, deform group, position), taps as a loop; columns are written as planes
// colT[bl][tap*C + c][p], rounded to tf32 (the grad_weight GEMM's B operand), exactly where dcn_im2col_planes_kernel puts them.
// X3: colT gets tf32(col) and colT_lo the remainder tf32(col - tf32(col)) at the same index (3-pass GEMM operand planes).
// DynAggSrc: goff as in dcn_bwd_coord_nhwc_kernel.
template <bool X3, class Src>
__device__ __forceinline__ void
dcn_bwd_coord_cols(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                          const Src& src) {
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG;
    const size_t total = (size_t)nb * s.DG * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int dgi = (idx / P) % s.DG;
        const int bl = idx / ((size_t)P * s.DG);
        const int b = b0 + bl;
        const int oy = p / s.Wo, ox = p - oy * s.Wo;
        const float* xb = xt + (size_t)b * s.H * s.W * s.C + dgi * cdg;
        for (int tap = 0; tap < K; ++tap) {
            const int ti = tap / s.kw, tj = tap - ti * s.kw;
            size_t ob, mb;
            float y, x, m;
            if constexpr (kDynAgg<Src>) {
                ob = dynagg_point(offset, src, s, b, dgi, tap, oy, ox, y, x, m, mb);
            } else {
                ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
                mb = ((size_t)(b * s.DG + dgi) * K + tap) * P + p;
                y = (float)(oy * s.sh - s.ph + ti * s.dh) + __ldcs(offset + ob);
                x = (float)(ox * s.sw - s.pw + tj * s.dw) + __ldcs(offset + ob + P);
                m = mask ? __ldcs(mask + mb) : 1.f;
            }
            float dy = 0.f, dx = 0.f, dm = 0.f;
            const size_t ct_off = ((size_t)bl * K * s.C + (size_t)tap * s.C + dgi * cdg) * P + p;
            float* ct = colT + ct_off;
            if (y > -1.f && x > -1.f && y < (float)s.H && x < (float)s.W) {
                const float fy0 = floorf(y), fx0 = floorf(x);
                const int y0 = (int)fy0, x0 = (int)fx0;
                const float ly = y - fy0, lx = x - fx0, hy = 1.f - ly, hx = 1.f - lx;
                const bool ty0 = y0 >= 0, ty1 = y0 + 1 <= s.H - 1, tx0 = x0 >= 0, tx1 = x0 + 1 <= s.W - 1;
                const int yc = ty0 ? y0 : 0, xc = tx0 ? x0 : 0;
                const float* base = xb + ((size_t)yc * s.W + xc) * s.C;
                const size_t dxo = (tx0 && tx1) ? s.C : 0, dyo = (ty0 && ty1) ? (size_t)s.W * s.C : 0;
                const float va = (ty0 && tx0) ? 1.f : 0.f, vb = (ty0 && tx1) ? 1.f : 0.f, vc = (ty1 && tx0) ? 1.f : 0.f,
                            vd = (ty1 && tx1) ? 1.f : 0.f;
                const float w0 = va * hy * hx * m, w1 = vb * hy * lx * m, w2 = vc * ly * hx * m, w3 = vd * ly * lx * m;
                const float* gc = gcol + ((size_t)bl * s.C * K + (size_t)dgi * cdg * K + tap) * P + p;
                for (int c0 = 0; c0 < cdg; c0 += 8) {
                    const Col8 v0 = ldg_col8(base + c0), v1 = ldg_col8(base + c0 + dxo), v2 = ldg_col8(base + c0 + dyo),
                               v3 = ldg_col8(base + c0 + dyo + dxo);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float a = va * v0.v[e], bq = vb * v1.v[e], cq = vc * v2.v[e], d = vd * v3.v[e];
                        const float g = __ldcs(gc + (size_t)(c0 + e) * K * P);
                        const float v = hy * hx * a + hy * lx * bq + ly * hx * cq + ly * lx * d;
                        dm += g * v;
                        dy += g * m * (hx * (cq - a) + lx * (d - bq));
                        dx += g * m * (hy * (bq - a) + ly * (d - cq));
                        // the column exactly as dcn_im2col_planes_kernel computes it (mask and validity folded into the weights)
                        const float col = w0 * v0.v[e] + w1 * v1.v[e] + w2 * v2.v[e] + w3 * v3.v[e], hi = to_tf32(col);
                        __stcs(ct + (size_t)(c0 + e) * P, hi);
                        if (X3) __stcs(colT_lo + ct_off + (size_t)(c0 + e) * P, to_tf32(col - hi));
                    }
                }
            } else {
                for (int c = 0; c < cdg; ++c) {
                    __stcs(ct + (size_t)c * P, 0.f);
                    if (X3) __stcs(colT_lo + ct_off + (size_t)c * P, 0.f);
                }
            }
            __stcs(goff + ob, dy);
            __stcs(goff + ob + P, dx);
            if constexpr (kDynAgg<Src>) __stcs(goff + mb, dm * m * (1.f - m));
            else if (gmask) __stcs(gmask + mb, dm);
        }
    }
}

template <bool X3>
__global__ void __launch_bounds__(256, 3)
dcn_bwd_coord_cols_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                          const PlaneSrc src) {
    dcn_bwd_coord_cols<X3>(xt, offset, mask, gcol, goff, gmask, colT, s, b0, nb, colT_lo, src);
}

template <bool X3>
__global__ void __launch_bounds__(256, 3)
dcn_bwd_coord_cols_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                          const float* __restrict__ gcol, float* __restrict__ goff, float* __restrict__ gmask,
                          float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                          const DynAggSrc src) {
    dcn_bwd_coord_cols<X3>(xt, offset, mask, gcol, goff, gmask, colT, s, b0, nb, colT_lo, src);
}

// written as planes colT[bl][tap*C + c][p] (k = position contiguous: the B operand of the
// tcgen05 grad_weight GEMM).  Lanes = consecutive positions, so each of the 8 scalar stores of a thread is a coalesced
// 128-byte warp store into its channel plane.  X3: colT_lo receives the tf32 remainders (as in dcn_bwd_coord_cols_kernel).
template <bool X3, class Src>
__device__ __forceinline__ void
dcn_im2col_planes(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                         float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                         const Src& src) {
    // thread = (bl, 8-channel chunk, position), taps as a loop (their corners meet in L1, as in the coordinate kernel)
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cdg = s.C / s.DG, C8 = s.C >> 3;
    const size_t total = (size_t)nb * C8 * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int j = (idx / P) % C8;
        const int bl = idx / ((size_t)P * C8);
        const int b = b0 + bl, c0 = j * 8, dgi = c0 / cdg;
        const int oy = p / s.Wo, ox = p - oy * s.Wo;
        const float* xb = xt + (size_t)b * s.H * s.W * s.C + c0;
        for (int tap = 0; tap < K; ++tap) {
            const int ti = tap / s.kw, tj = tap - ti * s.kw;
            float y, x, m;
            if constexpr (kDynAgg<Src>) {
                size_t mc;
                dynagg_point(offset, src, s, b, dgi, tap, oy, ox, y, x, m, mc);
            } else {
                const size_t ob = ((size_t)(b * s.DG + dgi) * 2 * K + 2 * tap) * P + p;
                y = (float)(oy * s.sh - s.ph + ti * s.dh) + __ldg(offset + ob);
                x = (float)(ox * s.sw - s.pw + tj * s.dw) + __ldg(offset + ob + P);
                m = mask ? __ldg(mask + ((size_t)(b * s.DG + dgi) * K + tap) * P + p) : 1.f;
            }
            float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (y > -1.f && x > -1.f && y < (float)s.H && x < (float)s.W) {
                const float fy0 = floorf(y), fx0 = floorf(x);
                const int y0 = (int)fy0, x0 = (int)fx0;
                const float ly = y - fy0, lx = x - fx0, hy = 1.f - ly, hx = 1.f - lx;
                const bool ty0 = y0 >= 0, ty1 = y0 + 1 <= s.H - 1, tx0 = x0 >= 0, tx1 = x0 + 1 <= s.W - 1;
                const int yc = ty0 ? y0 : 0, xc = tx0 ? x0 : 0;
                const float* base = xb + ((size_t)yc * s.W + xc) * s.C;
                const size_t dxo = (tx0 && tx1) ? s.C : 0, dyo = (ty0 && ty1) ? (size_t)s.W * s.C : 0;
                const float w0 = (ty0 && tx0) ? hy * hx * m : 0.f, w1 = (ty0 && tx1) ? hy * lx * m : 0.f;
                const float w2 = (ty1 && tx0) ? ly * hx * m : 0.f, w3 = (ty1 && tx1) ? ly * lx * m : 0.f;
                const Col8 v0 = ldg_col8(base), v1 = ldg_col8(base + dxo), v2 = ldg_col8(base + dyo), v3 = ldg_col8(base + dyo + dxo);
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = w0 * v0.v[e] + w1 * v1.v[e] + w2 * v2.v[e] + w3 * v3.v[e];
            }
            const size_t d_off = ((size_t)bl * K * s.C + (size_t)tap * s.C + c0) * P + p;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float hi = to_tf32(o[e]);              // GEMM operand: the tensor core's read truncates
                __stcs(colT + d_off + (size_t)e * P, hi);
                if (X3) __stcs(colT_lo + d_off + (size_t)e * P, to_tf32(o[e] - hi));
            }
        }
    }
}

template <bool X3>
__global__ void __launch_bounds__(256)
dcn_im2col_planes_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                         float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                         const PlaneSrc src) {
    dcn_im2col_planes<X3>(xt, offset, mask, colT, s, b0, nb, colT_lo, src);
}

template <bool X3>
__global__ void __launch_bounds__(256)
dcn_im2col_planes_kernel(const float* __restrict__ xt, const float* __restrict__ offset, const float* __restrict__ mask,
                         float* __restrict__ colT, const DcnShape s, int b0, int nb, float* __restrict__ colT_lo,
                         const DynAggSrc src) {
    dcn_im2col_planes<X3>(xt, offset, mask, colT, s, b0, nb, colT_lo, src);
}

// (wT_lo / dst_lo non-NULL: also the tf32 remainder, the lo plane of a 3-pass GEMM operand)
__global__ void dcn_weight_transpose_kernel(const float* __restrict__ w, float* __restrict__ wT, int Co, int MK,
                                            float* __restrict__ wT_lo) {
    const int total = Co * MK;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int oc = i % Co, m = i / Co;
        const float v = __ldg(w + (size_t)oc * MK + m), hi = to_tf32(v);
        wT[i] = hi;
        if (wT_lo) wT_lo[i] = to_tf32(v - hi);
    }
}

// tf32-rounded copy (GEMM operand whose natural layout is already the one the GEMM wants)
__global__ void dcn_round_tf32_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t n,
                                      float* __restrict__ dst_lo) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = __ldg(src + i), hi = to_tf32(v);
        dst[i] = hi;
        if (dst_lo) dst_lo[i] = to_tf32(v - hi);
    }
}

// gwT[i] += sum over the splits of part[s][i], in split order (deterministic)
__global__ void dcn_split_sum_kernel(const float* __restrict__ part, float* __restrict__ gwT, int n, int splits) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float a = gwT[i];
        for (int sp = 0; sp < splits; ++sp) a += part[(size_t)sp * n + i];
        gwT[i] = a;
    }
}

// grad_weight[oc][c][tap] += gwT[oc][tap*C + c]   (the grad_weight GEMM works in the tap-major column order)
__global__ void dcn_gw_permute_add_kernel(const float* __restrict__ gwT, float* __restrict__ gw, int Co, int C, int K) {
    const int total = Co * C * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int tap = i % K, c = (i / K) % C, oc = i / (K * C);
        gw[i] += gwT[((size_t)oc * K + tap) * C + c];
    }
}

// (4b) grad_weight[oc][m] += sum_{bl, p} gout[b][oc][p] * col[bl][m][p]   (deform_conv_cuda.cpp:659-664)
// grid (G * ceil(MK/64), ceil(opg/64), nb * pchunks), block 256; split-K partial sums merged with atomicAdd.
constexpr int WCHUNK = 2048;
__global__ void __launch_bounds__(256)
dcn_bwd_weight_kernel(const float* __restrict__ gout, const float* __restrict__ col, float* __restrict__ gw,
                      const DcnShape s, int b0, int pchunks) {
    __shared__ float As[DK][DT + 4];
    __shared__ float Bs[DK][DT + 4];
    const int K = s.kh * s.kw, P = s.Ho * s.Wo, cpg = s.C / s.G, opg = s.Co / s.G, MK = cpg * K;
    const int mt_per = cdiv_d(MK, DT);
    const int gi = blockIdx.x / mt_per, m0 = (blockIdx.x % mt_per) * DT, oc0 = blockIdx.y * DT;
    const int bl = blockIdx.z / pchunks, pc = blockIdx.z % pchunks, b = b0 + bl;
    const int pbeg = pc * WCHUNK, pend = min(P, pbeg + WCHUNK);
    const int t = threadIdx.x, lr = t >> 2, lk = (t & 3) * 4, ty = t >> 4, tx = t & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int oc = oc0 + lr, m = m0 + lr;
    const float* arow = (oc < opg) ? gout + ((size_t)b * s.Co + gi * opg + oc) * P : nullptr;
    const float* brow = (m < MK) ? col + ((size_t)bl * s.C * K + (size_t)gi * MK + m) * P : nullptr;
    for (int k0 = pbeg; k0 < pend; k0 += DK) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int pp = k0 + lk + e;
            As[lk + e][lr] = (arow && pp < pend) ? __ldg(arow + pp) : 0.f;
            Bs[lk + e][lr] = (brow && pp < pend) ? __ldg(brow + pp) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < DK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 bb = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int o = oc0 + ty * 4 + i;
        if (o >= opg) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int mm = m0 + tx * 4 + j;
            if (mm < MK) atomicAdd(gw + (size_t)(gi * opg + o) * MK + mm, acc[i][j]);
        }
    }
}

// (5) grad_bias[oc] += sum_{b, p} gout[b][oc][p]   (deform_conv_cuda.cpp:665-671); grid (Co, batch split), the
// partial sums of a channel are merged with one atomicAdd per block
__global__ void dcn_bwd_bias_kernel(const float* __restrict__ gout, float* __restrict__ gb, int B, int Co, int P) {
    __shared__ float red[32];
    const int oc = blockIdx.x;
    float sum = 0.f;
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
        const float* g = gout + ((size_t)b * Co + oc) * P;
        for (int p = threadIdx.x; p < P; p += blockDim.x) sum += g[p];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) atomicAdd(gb + oc, v);
    }
}

// =====================================================================================================
// DynAgg glue (ref_mrapa_restoration_arch.py:55-73): chunk / cat / pre-offset add / sigmoid in one pass
// =====================================================================================================
__global__ void dynagg_offsets_kernel(const float* __restrict__ conv_out, const float* __restrict__ pre,
                                      float* __restrict__ offset, float* __restrict__ mask,
                                      float* __restrict__ abs_sum, int B, int dg, int K, int P) {
    const int OC = 2 * dg * K, MC = dg * K, TC = OC + MC;
    const size_t total = (size_t)B * TC * P;
    float local = 0.f;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int ch = (idx / P) % TC;
        const int b = idx / ((size_t)P * TC);
        const float v = conv_out[idx];
        if (ch < OC) {
            // offset channel ch: tap k = (ch/2) % K; even = y (pre[...,1]), odd = x (pre[...,0])
            const int k = (ch >> 1) % K;
            const float pv = pre[(((size_t)b * K + k) * P + p) * 2 + ((ch & 1) ? 0 : 1)];
            offset[((size_t)b * OC + ch) * P + p] = v + pv;
            local += fabsf(v);
        } else {
            mask[((size_t)b * MC + (ch - OC)) * P + p] = 1.f / (1.f + expf(-v));
        }
    }
    if (abs_sum) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
        if ((threadIdx.x & 31) == 0 && local != 0.f) atomicAdd(abs_sum, local);
    }
}

// The same pass, four positions per thread (16-byte accesses, no integer division in the loop): grid.y = (sample, plane).
// Same arithmetic per element as the scalar kernel; used when P % 4 == 0 and the tensors are 16-byte aligned.
__global__ void __launch_bounds__(256)
dynagg_offsets_vec4_kernel(const float* __restrict__ conv_out, const float* __restrict__ pre, float* __restrict__ offset,
                           float* __restrict__ mask, float* __restrict__ abs_sum, int dg, int K, int P) {
    const int OC = 2 * dg * K, MC = dg * K, TC = OC + MC;
    const int b = blockIdx.y / TC, ch = blockIdx.y - b * TC;
    const float4* src = reinterpret_cast<const float4*>(conv_out + ((size_t)b * TC + ch) * P);
    const int P4 = P >> 2;
    float local = 0.f;
    if (ch < OC) {
        const int k = (ch >> 1) % K;
        const int comp = (ch & 1) ? 0 : 1;       // even plane = y = pre[..., 1], odd plane = x = pre[..., 0]
        const float4* pv = reinterpret_cast<const float4*>(pre + ((size_t)b * K + k) * P * 2);   // (x, y) pairs of 2 positions
        float4* dst = reinterpret_cast<float4*>(offset + ((size_t)b * OC + ch) * P);
        // two float4 per thread and iteration: six independent 16-byte loads in flight (the pass is HBM-bound)
        const int step = gridDim.x * blockDim.x;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P4; i += 2 * step) {
            const int i2 = i + step;
            const bool two = i2 < P4;
            const float4 v = __ldcs(src + i);
            const float4 p0 = __ldg(pv + 2 * i), p1 = __ldg(pv + 2 * i + 1);
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f), q0 = w, q1 = w;
            if (two) {
                w = __ldcs(src + i2);
                q0 = __ldg(pv + 2 * i2);
                q1 = __ldg(pv + 2 * i2 + 1);
            }
            const float a0 = comp ? p0.y : p0.x, a1 = comp ? p0.w : p0.z, a2 = comp ? p1.y : p1.x, a3 = comp ? p1.w : p1.z;
            __stcs(dst + i, make_float4(v.x + a0, v.y + a1, v.z + a2, v.w + a3));
            local += fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(v.w);
            if (two) {
                const float b0 = comp ? q0.y : q0.x, b1 = comp ? q0.w : q0.z, b2 = comp ? q1.y : q1.x, b3 = comp ? q1.w : q1.z;
                __stcs(dst + i2, make_float4(w.x + b0, w.y + b1, w.z + b2, w.w + b3));
                local += fabsf(w.x) + fabsf(w.y) + fabsf(w.z) + fabsf(w.w);
            }
        }
    } else {
        float4* dst = reinterpret_cast<float4*>(mask + ((size_t)b * MC + (ch - OC)) * P);
        const int step = gridDim.x * blockDim.x;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P4; i += 2 * step) {
            const int i2 = i + step;
            const bool two = i2 < P4;
            const float4 v = __ldcs(src + i);
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
            if (two) w = __ldcs(src + i2);
            __stcs(dst + i, make_float4(1.f / (1.f + expf(-v.x)), 1.f / (1.f + expf(-v.y)), 1.f / (1.f + expf(-v.z)),
                                        1.f / (1.f + expf(-v.w))));
            if (two)
                __stcs(dst + i2, make_float4(1.f / (1.f + expf(-w.x)), 1.f / (1.f + expf(-w.y)), 1.f / (1.f + expf(-w.z)),
                                             1.f / (1.f + expf(-w.w))));
        }
    }
    if (abs_sum) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
        if ((threadIdx.x & 31) == 0 && local != 0.f) atomicAdd(abs_sum, local);
    }
}

// Backward of the glue: grad of the raw conv_offset_mask output = [grad_offset, grad_mask * m * (1 - m)] (the pre-offsets are
// constants; d sigmoid = m (1 - m)), one pass with 16-byte accesses instead of torch's mul / mul / cat.  grid.y = (sample, plane).
__global__ void __launch_bounds__(256)
dynagg_offsets_bwd_vec4_kernel(const float* __restrict__ g_offset, const float* __restrict__ g_mask,
                               const float* __restrict__ mask, float* __restrict__ g_conv, int dg, int K, int P) {
    const int OC = 2 * dg * K, MC = dg * K, TC = OC + MC;
    const int b = blockIdx.y / TC, ch = blockIdx.y - b * TC;
    float4* dst = reinterpret_cast<float4*>(g_conv + ((size_t)b * TC + ch) * P);
    const int P4 = P >> 2;
    if (ch < OC) {
        const float4* src = reinterpret_cast<const float4*>(g_offset + ((size_t)b * OC + ch) * P);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P4; i += gridDim.x * blockDim.x) dst[i] = __ldcs(src + i);
    } else {
        const float4* gm = reinterpret_cast<const float4*>(g_mask + ((size_t)b * MC + (ch - OC)) * P);
        const float4* mk = reinterpret_cast<const float4*>(mask + ((size_t)b * MC + (ch - OC)) * P);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P4; i += gridDim.x * blockDim.x) {
            const float4 g = __ldcs(gm + i), m = __ldcs(mk + i);
            dst[i] = make_float4(g.x * m.x * (1.f - m.x), g.y * m.y * (1.f - m.y), g.z * m.z * (1.f - m.z),
                                 g.w * m.w * (1.f - m.w));
        }
    }
}
__global__ void dynagg_offsets_bwd_kernel(const float* __restrict__ g_offset, const float* __restrict__ g_mask,
                                          const float* __restrict__ mask, float* __restrict__ g_conv, int B, int dg, int K,
                                          int P) {
    const int OC = 2 * dg * K, MC = dg * K, TC = OC + MC;
    const size_t total = (size_t)B * TC * P;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int p = idx % P;
        const int ch = (idx / P) % TC;
        const int b = idx / ((size_t)P * TC);
        if (ch < OC) {
            g_conv[idx] = g_offset[((size_t)b * OC + ch) * P + p];
        } else {
            const size_t mi = ((size_t)b * MC + (ch - OC)) * P + p;
            const float m = mask[mi];
            g_conv[idx] = g_mask[mi] * m * (1.f - m);
        }
    }
}

// =====================================================================================================
// host side
// =====================================================================================================
int dcn_make_shape(DcnShape* s, int B, int C, int H, int W, int Co, int kh, int kw, int sh, int sw, int ph, int pw,
                   int dh, int dw, int G, int DG) {
    MREFSR_CHECK(B > 0 && C > 0 && H > 0 && W > 0 && Co > 0 && kh > 0 && kw > 0, ERR_BAD_ARG, "dcn: bad sizes");
    MREFSR_CHECK(sh > 0 && sw > 0 && dh > 0 && dw > 0 && ph >= 0 && pw >= 0, ERR_BAD_ARG, "dcn: bad stride/pad/dilation");
    MREFSR_CHECK(G > 0 && DG > 0 && C % G == 0 && Co % G == 0, ERR_BAD_ARG,
                 "dcn: input shape and kernel channels won't match: (%d vs %d groups)", C, G);
    MREFSR_CHECK(C % DG == 0, ERR_BAD_ARG, "dcn: channels %d not divisible by deformable_group %d", C, DG);
    s->B = B; s->C = C; s->H = H; s->W = W; s->Co = Co; s->kh = kh; s->kw = kw; s->sh = sh; s->sw = sw;
    s->ph = ph; s->pw = pw; s->dh = dh; s->dw = dw; s->G = G; s->DG = DG;
    s->Ho = (H + 2 * ph - (dh * (kh - 1) + 1)) / sh + 1;
    s->Wo = (W + 2 * pw - (dw * (kw - 1) + 1)) / sw + 1;
    MREFSR_CHECK(s->Ho > 0 && s->Wo > 0, ERR_BAD_ARG, "dcn: empty output %d x %d", s->Ho, s->Wo);
    return 0;
}

constexpr int BWD_MAX_SPLITS = 32;     // split-K pieces of the grad_weight GEMM (partial sums in the workspace)

static int bwd_chunk(const DcnShape& s, bool x3) {
    const size_t per = (size_t)s.C * s.kh * s.kw * s.Ho * s.Wo * 4;
    // two scratch tensors of <= 1 GiB (columns, their gradient): fewer, larger launches.  The 3-pass mode adds the
    // columns' lo plane and keeps the three within the same 2 GiB.
    size_t nb = (x3 ? ((size_t)2048 << 20) / 3 : ((size_t)1024 << 20)) / per;
    if (nb < 1) nb = 1;
    if (nb > (size_t)s.B) nb = s.B;
    return (int)nb;
}

static int grid_for(size_t total) {
    size_t blocks = (total + 255) / 256;
    const size_t cap = (size_t)sm_count() * 32;
    return (int)(blocks > cap ? cap : blocks);
}

// The DCN backward's host body for either sample source (PlaneSrc / DynAggSrc, dcn_common.cuh): the chunk loop over
// samples, the two GEMMs (tcgen05 or CUDA cores) and grad_weight's split-K sums.  DynAggSrc: `offset` is the raw
// conv_offset_mask output, `mask` is unused, grad_offset receives the gradient of that output, grad_mask is NULL, and
// the caller has checked that the shape takes the NHWC coordinate kernels (mrefsr_dynagg_dcn_backward).
template <class Src>
static int dcn_backward(const float* input, const float* weight, const float* offset, const float* mask,
                        const float* grad_output, float* grad_input, float* grad_weight, float* grad_bias,
                        float* grad_offset, float* grad_mask, const DcnShape& s, int with_bias, int mode, void* workspace,
                        size_t workspace_bytes, cudaStream_t st, const Src& src) {
    const int B = s.B, C = s.C, H = s.H, W = s.W, Co = s.Co, kh = s.kh, kw = s.kw, group = s.G, deformable_group = s.DG;
    // MREFSR_DCN_FP32: exact-fp32 CUDA-core GEMMs of this file; otherwise the two plain GEMMs run on tcgen05
    // (gemm_tc.cu, TF32 operands, fp32 accumulate) whenever the operand pitches allow TMA (group 1, Co % 4 == 0 for
    // the columns GEMM, output positions % 4 == 0 for the grad_weight GEMM)
    const bool tc_gemm = mode != MREFSR_DCN_FP32;
    // MREFSR_DCN_TF32X3: those two GEMMs take hi / lo operand planes and run the 3-pass kernel (fp32-grade products)
    const bool x3 = mode == MREFSR_DCN_TF32X3;
    int rc = 0;
    const int K = kh * kw, P = s.Ho * s.Wo, cpg = C / group, opg = Co / group, MK = cpg * K;
    const int nbmax = bwd_chunk(s, x3);
    const size_t buf = align_up((size_t)nbmax * C * K * P * 4, 1024);
    const size_t xt_bytes = align_up((size_t)B * C * H * W * 4, 1024), gwt_bytes = align_up((size_t)Co * C * K * 4, 1024);
    const size_t got_bytes = align_up((size_t)B * Co * P * 4, 1024);
    const size_t part_bytes = align_up((size_t)BWD_MAX_SPLITS * Co * C * K * 4, 1024);
    const bool small_enough = (size_t)B * C * H * W < ((size_t)1 << 31) && (size_t)B * Co * P < ((size_t)1 << 31);
    // columns GEMM on tcgen05: gcol[bl] (MK x P) = W^T (MK x Co) . gout[b] (Co x P); B operand = gout position-major
    const bool tc_gcol = tc_gemm && (grad_input || grad_offset) && group == 1 && Co % 4 == 0 && small_enough;
    // grad_weight GEMM on tcgen05: gwT (Co x K*C, tap-major) += gout[b] (Co x P) . colT[bl]^T, k = positions
    const bool tc_gw = tc_gemm && grad_weight && group == 1 && C % 8 == 0 && (C / deformable_group) % 8 == 0 && P % 4 == 0 &&
                       small_enough;
    const size_t need = 2 * buf + xt_bytes + 2 * got_bytes + 2 * gwt_bytes + part_bytes;
    const size_t need_all = need + (x3 ? buf + 2 * got_bytes + gwt_bytes : 0);
    MREFSR_CHECK(workspace && workspace_bytes >= need_all, ERR_WORKSPACE, "dcn backward: workspace too small (%zu < %zu)",
                 workspace_bytes, need_all);
    MREFSR_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, ERR_WORKSPACE, "dcn backward: workspace must be 1024-byte aligned");
    uint8_t* wsp = static_cast<uint8_t*>(workspace);
    float* gcol = reinterpret_cast<float*>(wsp);
    float* col = reinterpret_cast<float*>(wsp + buf);
    float* xt = reinterpret_cast<float*>(wsp + 2 * buf);
    float* goutT = reinterpret_cast<float*>(wsp + 2 * buf + xt_bytes);
    float* gwT = reinterpret_cast<float*>(wsp + 2 * buf + xt_bytes + got_bytes);
    float* wT = reinterpret_cast<float*>(wsp + 2 * buf + xt_bytes + got_bytes + gwt_bytes);
    float* part = reinterpret_cast<float*>(wsp + 2 * buf + xt_bytes + got_bytes + 2 * gwt_bytes);
    float* goutR = reinterpret_cast<float*>(wsp + 2 * buf + xt_bytes + got_bytes + 2 * gwt_bytes + part_bytes);
    // lo planes of the 3-pass GEMM operands, after the buffers above (counted by mrefsr_dcn_workspace_bytes for mode 3)
    uint8_t* lo_base = wsp + need;
    float* col_lo = x3 ? reinterpret_cast<float*>(lo_base) : nullptr;
    float* goutT_lo = x3 ? reinterpret_cast<float*>(lo_base + buf) : nullptr;
    float* goutR_lo = x3 ? reinterpret_cast<float*>(lo_base + buf + got_bytes) : nullptr;
    float* wT_lo = x3 ? reinterpret_cast<float*>(lo_base + buf + 2 * got_bytes) : nullptr;
    // grad_offset / grad_mask from the NHWC copy (four 256-bit corner loads per 8-channel chunk instead of 32 scalar loads)
    const bool nhwc_coord = tc_gemm && grad_offset && C % 8 == 0 && (C / deformable_group) % 8 == 0 && small_enough;
    if ((tc_gw || nhwc_coord) && src_nhwc(src)) {
        xt = const_cast<float*>(input);             // the caller's NHWC input already is the gather layout
    } else if (tc_gw || nhwc_coord) {
        rc = dcn_nchw_to_nhwc(input, xt, B, C, H * W, st);
        if (rc) return rc;
    }
    if (tc_gw) {
        MREFSR_CUDA(cudaMemsetAsync(gwT, 0, (size_t)Co * C * K * 4, st));
        dcn_round_tf32_kernel<<<grid_for((size_t)B * Co * P), 256, 0, st>>>(grad_output, goutR, (size_t)B * Co * P, goutR_lo);
        MREFSR_LAUNCH_CHECK();
        count_launches(1);
    }
    if (tc_gcol) {
        rc = dcn_nchw_to_nhwc(grad_output, goutT, B, Co, P, st, true, goutT_lo);
        if (rc) return rc;
        dcn_weight_transpose_kernel<<<cdiv(Co * MK, 256), 256, 0, st>>>(weight, wT, Co, MK, wT_lo);
        MREFSR_LAUNCH_CHECK();
        count_launches(1);
    }
    if (grad_input) MREFSR_CUDA(cudaMemsetAsync(grad_input, 0, (size_t)B * C * H * W * 4, st));
    for (int b0 = 0; b0 < B; b0 += nbmax) {
        const int nb = (B - b0 < nbmax) ? B - b0 : nbmax;
        if (tc_gcol) {
            // (deform_conv_cuda.cpp:623-626), all samples of the chunk in one launch
            rc = gemm_tf32_nt(wT, Co, 0, goutT + (size_t)b0 * P * Co, Co, (long long)P * Co, gcol, P, (long long)MK * P, MK, P,
                              Co, nb, 0, 1, st, wT_lo, x3 ? goutT_lo + (size_t)b0 * P * Co : nullptr);
            if (rc) return rc;
        } else if (grad_input || grad_offset) {
            dcn_bwd_gcol_kernel<<<dim3(cdiv(P, DT), group * cdiv(MK, DT), nb), 256, 0, st>>>(weight, grad_output, gcol, s, b0);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        }
        // coordinate gradients and recomputed columns from ONE gather when the backward wants both
        const bool merged = grad_offset && nhwc_coord && tc_gw;
        if (merged) {
            if (x3)
                dcn_bwd_coord_cols_kernel<true><<<grid_for((size_t)nb * deformable_group * P), 256, 0, st>>>(
                    xt, offset, mask, gcol, grad_offset, grad_mask, col, s, b0, nb, col_lo, src);
            else
                dcn_bwd_coord_cols_kernel<false><<<grid_for((size_t)nb * deformable_group * P), 256, 0, st>>>(
                    xt, offset, mask, gcol, grad_offset, grad_mask, col, s, b0, nb, nullptr, src);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        } else if (grad_offset && nhwc_coord) {
            dcn_bwd_coord_nhwc_kernel<<<grid_for((size_t)nb * deformable_group * P), 256, 0, st>>>(
                xt, offset, mask, gcol, grad_offset, grad_mask, s, b0, nb, src);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        } else if (grad_offset) {
            MREFSR_CHECK(!kDynAgg<Src>, ERR_UNSUPPORTED, "dynagg backward: no planar coordinate kernel");
            dcn_bwd_coord_kernel<<<grid_for((size_t)nb * deformable_group * K * P), 256, 0, st>>>(
                input, offset, mask, gcol, grad_offset, grad_mask, s, b0, nb);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        }
        if (grad_input) {
            dcn_bwd_input_kernel<<<grid_for((size_t)nb * C * K * P), 256, 0, st>>>(offset, mask, gcol, grad_input, s, b0, nb,
                                                                                      src);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        }
        if (tc_gw) {
            // recomputed columns (deform_conv_cuda.cpp:647-650) as planes colT[bl][tap*C + c][p], then the chunk's share
            // of grad_weight (:659-664) as one split-K GEMM whose partial sums are added up in a fixed order
            if (!merged) {
                if (x3)
                    dcn_im2col_planes_kernel<true><<<grid_for((size_t)nb * (C / 8) * P), 256, 0, st>>>(
                        xt, offset, mask, col, s, b0, nb, col_lo, src);
                else
                    dcn_im2col_planes_kernel<false><<<grid_for((size_t)nb * (C / 8) * P), 256, 0, st>>>(
                        xt, offset, mask, col, s, b0, nb, nullptr, src);
                MREFSR_LAUNCH_CHECK();
                count_launches(1);
            }
            const long long all_kb = (long long)nb * cdiv(P, 32);
            const int tiles = cdiv(Co, 128) * cdiv(K * C, 128);
            int splits = cdiv(2 * sm_count(), tiles);
            if (splits > BWD_MAX_SPLITS) splits = BWD_MAX_SPLITS;
            if (splits > all_kb) splits = (int)all_kb;
            if (splits < 1) splits = 1;
            rc = gemm_tf32_nt(goutR + (size_t)b0 * Co * P, P, (long long)Co * P, col, P, (long long)K * C * P, part, K * C,
                              (long long)Co * K * C, Co, K * C, P, nb, 1, splits, st,
                              x3 ? goutR_lo + (size_t)b0 * Co * P : nullptr, col_lo);
            if (rc) return rc;
            dcn_split_sum_kernel<<<cdiv(Co * C * K, 256), 256, 0, st>>>(part, gwT, Co * C * K, splits);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        } else if (grad_weight) {
            dcn_im2col_kernel<<<grid_for((size_t)nb * C * K * P), 256, 0, st>>>(input, offset, mask, col, s, b0, nb, src);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
            const int pchunks = cdiv(P, WCHUNK);
            dcn_bwd_weight_kernel<<<dim3(group * cdiv(MK, DT), cdiv(opg, DT), nb * pchunks), 256, 0, st>>>(
                grad_output, col, grad_weight, s, b0, pchunks);
            MREFSR_LAUNCH_CHECK();
            count_launches(1);
        }
    }
    if (tc_gw) {
        dcn_gw_permute_add_kernel<<<cdiv(Co * C * K, 256), 256, 0, st>>>(gwT, grad_weight, Co, C, K);
        MREFSR_LAUNCH_CHECK();
        count_launches(1);
    }
    if (with_bias) {
        dcn_bwd_bias_kernel<<<dim3(Co, B < 32 ? B : 32), 256, 0, st>>>(grad_output, grad_bias, B, Co, P);
        MREFSR_LAUNCH_CHECK();
        count_launches(1);
    }
    return 0;
}

int dcn_forward_fp32(const float* x, const float* w, const float* bias, const float* off, const float* mask, float* out,
                     const DcnShape& s, cudaStream_t st) {
    const int P = s.Ho * s.Wo, opg = s.Co / s.G;
    dim3 grid(cdiv(P, DT), s.G * cdiv(opg, DT), s.B);
    ScopedTiming tm(MREFSR_K_DCN_FWD, st);
    dcn_fwd_simt_kernel<<<grid, 256, 0, st>>>(x, off, mask, w, bias, out, s);
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

}  // namespace mrefsr

using namespace mrefsr;

extern "C" {

int mrefsr_dcn_tile_plan(int B, int Ho, int Wo, int* meta, int* coords, size_t max_rows) {
    MREFSR_CHECK(B > 0 && Ho > 0 && Wo > 0 && meta, ERR_BAD_ARG, "tile plan: bad arguments");
    MREFSR_CHECK((long long)B * Ho * Wo < (1ll << 31) - 256, ERR_BAD_ARG, "tile plan: too many positions");
    return dcn_tc_tile_plan(B, Ho, Wo, meta, coords, max_rows);
}

size_t mrefsr_dcn_workspace_bytes(int B, int C, int H, int W, int Co, int kh, int kw, int stride_h, int stride_w,
                                  int pad_h, int pad_w, int dil_h, int dil_w, int group, int deformable_group, int mode,
                                  int backward) {
    DcnShape s;
    if (dcn_make_shape(&s, B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, group,
                       deformable_group))
        return 0;
    if (backward) { // gcol + col chunks, NHWC copies of the input and of grad_output, W^T, tap-major grad_weight scratch
                    // and the split-K partial sums of the grad_weight GEMM; the 3-pass mode adds the lo planes of the
                    // GEMM operands (col, both copies of grad_output, W^T)
        const bool x3 = mode == MREFSR_DCN_TF32X3;
        const size_t buf = align_up((size_t)bwd_chunk(s, x3) * C * kh * kw * s.Ho * s.Wo * 4, 1024);
        const size_t got = align_up((size_t)B * Co * s.Ho * s.Wo * 4, 1024), gwt = align_up((size_t)Co * C * kh * kw * 4, 1024);
        return 2 * buf + align_up((size_t)B * C * H * W * 4, 1024) + 2 * got + 2 * gwt +
               align_up((size_t)BWD_MAX_SPLITS * Co * C * kh * kw * 4, 1024) + (x3 ? buf + 2 * got + gwt : 0) + 1024;
    }
    return dcn_tc_workspace_bytes(s, mode) + 1024;
}

int mrefsr_modulated_deform_conv_forward(const float* input, const float* weight, const float* bias,
                                         const float* offset, const float* mask, float* output, int B, int C, int H,
                                         int W, int Co, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w,
                                         int dil_h, int dil_w, int group, int deformable_group, int with_bias, int mode,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    MREFSR_CHECK(input && weight && offset && output, ERR_BAD_ARG, "dcn forward: null pointer argument");
    MREFSR_CHECK(!with_bias || bias, ERR_BAD_ARG, "dcn forward: with_bias set but bias is NULL");
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, group,
                            deformable_group);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float* bp = with_bias ? bias : nullptr;
    int m = mode;
    if (m == MREFSR_DCN_AUTO) m = dcn_tc_eligible(s) ? MREFSR_DCN_TF32 : MREFSR_DCN_FP32;
    if (m == MREFSR_DCN_FP32) return dcn_forward_fp32(input, weight, bp, offset, mask, output, s, st);
    MREFSR_CHECK(m == MREFSR_DCN_TF32 || m == MREFSR_DCN_TF32X3, ERR_BAD_ARG, "dcn forward: unknown mode %d", mode);
    MREFSR_CHECK(dcn_tc_eligible(s), ERR_UNSUPPORTED,
                 "dcn forward: tcgen05 path needs group 1, C %% 32 == 0, Co %% 32 == 0, Co <= 256, "
                 "(C/deformable_group) %% 4 == 0");
    return dcn_forward_tc(input, weight, bp, offset, mask, output, s, workspace, workspace_bytes, st,
                          m == MREFSR_DCN_TF32X3);
}

int mrefsr_modulated_deform_conv_backward(const float* input, const float* weight, const float* offset,
                                          const float* mask, const float* grad_output, float* grad_input,
                                          float* grad_weight, float* grad_bias, float* grad_offset, float* grad_mask,
                                          int B, int C, int H, int W, int Co, int kh, int kw, int stride_h, int stride_w,
                                          int pad_h, int pad_w, int dil_h, int dil_w, int group, int deformable_group,
                                          int with_bias, int mode, void* workspace, size_t workspace_bytes,
                                          void* stream) {
    MREFSR_CHECK(input && weight && offset && grad_output, ERR_BAD_ARG, "dcn backward: null pointer argument");
    MREFSR_CHECK(grad_offset || !grad_mask, ERR_BAD_ARG, "dcn backward: grad_mask requires grad_offset");
    MREFSR_CHECK(!with_bias || grad_bias, ERR_BAD_ARG, "dcn backward: with_bias set but grad_bias is NULL");
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, group,
                            deformable_group);
    if (rc) return rc;
    return dcn_backward(input, weight, offset, mask, grad_output, grad_input, grad_weight, grad_bias, grad_offset,
                        grad_mask, s, with_bias, mode, workspace, workspace_bytes, static_cast<cudaStream_t>(stream),
                        PlaneSrc{});
}

int mrefsr_gemm_tf32_nt(const float* A, int lda, long long a_batch_stride, const float* B, int ldb, long long b_batch_stride,
                        float* D, int ldd, long long d_stride, int M, int N, int K, int batch, int reduce, int splits,
                        void* stream) {
    MREFSR_CHECK(A && B && D, ERR_BAD_ARG, "gemm: null pointer argument");
    MREFSR_CHECK(!reduce || splits >= 1, ERR_BAD_ARG, "gemm: reduce mode needs splits >= 1");
    return gemm_tf32_nt(A, lda, a_batch_stride, B, ldb, b_batch_stride, D, ldd, d_stride, M, N, K, batch, reduce, splits,
                        static_cast<cudaStream_t>(stream));
}

int mrefsr_gemm_tf32x3_nt(const float* A_hi, const float* A_lo, int lda, long long a_batch_stride, const float* B_hi,
                          const float* B_lo, int ldb, long long b_batch_stride, float* D, int ldd, long long d_stride, int M,
                          int N, int K, int batch, int reduce, int splits, void* stream) {
    MREFSR_CHECK(A_hi && A_lo && B_hi && B_lo && D, ERR_BAD_ARG, "gemm (x3): null pointer argument");
    MREFSR_CHECK(!reduce || splits >= 1, ERR_BAD_ARG, "gemm (x3): reduce mode needs splits >= 1");
    return gemm_tf32_nt(A_hi, lda, a_batch_stride, B_hi, ldb, b_batch_stride, D, ldd, d_stride, M, N, K, batch, reduce,
                        splits, static_cast<cudaStream_t>(stream), A_lo, B_lo);
}

int mrefsr_dcn_pack_weights(const float* weight, float* packed, int Co, int C, int K, void* stream) {
    MREFSR_CHECK(weight && packed && Co > 0 && C > 0 && K > 0, ERR_BAD_ARG, "pack_weights: bad arguments");
    return dcn_pack_weights(weight, packed, Co, C, K, static_cast<cudaStream_t>(stream));
}

int mrefsr_dcn_pack_weights_x3(const float* weight, float* packed, int Co, int C, int K, void* stream) {
    MREFSR_CHECK(weight && packed && Co > 0 && C > 0 && K > 0, ERR_BAD_ARG, "pack_weights_x3: bad arguments");
    return dcn_pack_weights(weight, packed, Co, C, K, static_cast<cudaStream_t>(stream), true);
}

int mrefsr_dynagg_dcn_forward(const float* input, const float* weight, const float* bias, const float* conv_out,
                              const int64_t* max_idx, int flow_scale, float* output, int B, int C, int H, int W, int Co,
                              int deformable_group, int with_bias, void* workspace, size_t workspace_bytes,
                              void* stream) {
    MREFSR_CHECK(input && weight && conv_out && max_idx && output, ERR_BAD_ARG, "dynagg forward: null pointer argument");
    MREFSR_CHECK(!with_bias || bias, ERR_BAD_ARG, "dynagg forward: with_bias set but bias is NULL");
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, 3, 3, 1, 1, 1, 1, 1, 1, 1, deformable_group);
    if (rc) return rc;
    MREFSR_CHECK(dcn_tc_eligible(s), ERR_UNSUPPORTED,
                 "dynagg forward: needs C %% 32 == 0, (C/deformable_group) %% 8 == 0, Co %% 32 == 0, Co <= 256");
    return dcn_forward_tc_impl(input, weight, with_bias ? bias : nullptr, conv_out, nullptr,
                               reinterpret_cast<const long long*>(max_idx), flow_scale, output, s, workspace,
                               workspace_bytes, static_cast<cudaStream_t>(stream), 0, 1.f, nullptr);
}

int mrefsr_dynagg_dcn_forward_ex(const float* input, const float* weight, const float* bias, const float* conv_out,
                                 const int64_t* max_idx, int flow_scale, float* output, int B, int C, int H, int W,
                                 int Co, int deformable_group, int with_bias, int layout_flags, float out_slope,
                                 void* workspace, size_t workspace_bytes, void* stream) {
    MREFSR_CHECK(input && weight && conv_out && max_idx && output, ERR_BAD_ARG, "dynagg forward: null pointer argument");
    MREFSR_CHECK(!with_bias || bias, ERR_BAD_ARG, "dynagg forward: with_bias set but bias is NULL");
    MREFSR_CHECK((layout_flags & ~(MREFSR_DCN_IN_NHWC | MREFSR_DCN_OUT_NHWC | MREFSR_DCN_W_PACKED | MREFSR_DCN_X3)) == 0, ERR_BAD_ARG,
                 "dynagg forward: unknown layout flags 0x%x", layout_flags);
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, 3, 3, 1, 1, 1, 1, 1, 1, 1, deformable_group);
    if (rc) return rc;
    MREFSR_CHECK(dcn_tc_eligible(s), ERR_UNSUPPORTED,
                 "dynagg forward: needs C %% 32 == 0, (C/deformable_group) %% 8 == 0, Co %% 32 == 0, Co <= 256");
    return dcn_forward_tc_impl(input, weight, with_bias ? bias : nullptr, conv_out, nullptr,
                               reinterpret_cast<const long long*>(max_idx), flow_scale, output, s, workspace,
                               workspace_bytes, static_cast<cudaStream_t>(stream), layout_flags, out_slope, nullptr);
}

int mrefsr_dynagg_dcn_forward_multi(const float* input, const float* weight, const float* bias, const float* conv_out,
                                    const int64_t* max_idx, int flow_scale, float* const* outputs, int n_outputs,
                                    int dst_group, int dst_stride, int dst_offset, int B, int C, int H, int W, int Co,
                                    int deformable_group, int with_bias, int layout_flags, float out_slope,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    MREFSR_CHECK(input && weight && conv_out && max_idx && outputs, ERR_BAD_ARG, "dynagg forward: null pointer argument");
    MREFSR_CHECK(!with_bias || bias, ERR_BAD_ARG, "dynagg forward: with_bias set but bias is NULL");
    MREFSR_CHECK((layout_flags & ~(MREFSR_DCN_IN_NHWC | MREFSR_DCN_OUT_NHWC | MREFSR_DCN_W_PACKED | MREFSR_DCN_X3)) == 0, ERR_BAD_ARG,
                 "dynagg forward: unknown layout flags 0x%x", layout_flags);
    MREFSR_CHECK(n_outputs >= 1 && n_outputs <= 8, ERR_BAD_ARG, "dynagg forward: 1..8 output buffers (got %d)", n_outputs);
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, 3, 3, 1, 1, 1, 1, 1, 1, 1, deformable_group);
    if (rc) return rc;
    MREFSR_CHECK(dcn_tc_eligible(s), ERR_UNSUPPORTED,
                 "dynagg forward: needs C %% 32 == 0, (C/deformable_group) %% 8 == 0, Co %% 32 == 0, Co <= 256");
    DcnOutputs m;
    for (int k = 0; k < 8; ++k) m.ptr[k] = k < n_outputs ? outputs[k] : nullptr;
    m.n = n_outputs;
    m.group = dst_group;
    m.stride = dst_stride;
    m.offset = dst_offset;
    m.slab_rows = 0;
    return dcn_forward_tc_impl(input, weight, with_bias ? bias : nullptr, conv_out, nullptr,
                               reinterpret_cast<const long long*>(max_idx), flow_scale, nullptr, s, workspace,
                               workspace_bytes, static_cast<cudaStream_t>(stream), layout_flags, out_slope, &m);
}

int mrefsr_dynagg_dcn_forward_slabs(const float* input, const float* weight, const float* bias, const float* conv_out,
                                    const int64_t* max_idx, int flow_scale, float* const* outputs, int n_outputs,
                                    int slab_rows, int dst_group, int dst_stride, int dst_offset, int B, int C, int H,
                                    int W, int Co, int deformable_group, int with_bias, int layout_flags, float out_slope,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    MREFSR_CHECK(input && weight && conv_out && max_idx && outputs, ERR_BAD_ARG, "dynagg forward: null pointer argument");
    MREFSR_CHECK(!with_bias || bias, ERR_BAD_ARG, "dynagg forward: with_bias set but bias is NULL");
    MREFSR_CHECK((layout_flags & ~(MREFSR_DCN_IN_NHWC | MREFSR_DCN_W_PACKED | MREFSR_DCN_X3)) == 0, ERR_BAD_ARG,
                 "dynagg forward (slabs): unknown or unsupported layout flags 0x%x", layout_flags);
    MREFSR_CHECK(n_outputs >= 1 && n_outputs <= 8 && slab_rows >= 1, ERR_BAD_ARG,
                 "dynagg forward (slabs): 1..8 output buffers and slab_rows >= 1 (got %d, %d)", n_outputs, slab_rows);
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, 3, 3, 1, 1, 1, 1, 1, 1, 1, deformable_group);
    if (rc) return rc;
    MREFSR_CHECK(dcn_tc_eligible(s), ERR_UNSUPPORTED,
                 "dynagg forward: needs C %% 32 == 0, (C/deformable_group) %% 8 == 0, Co %% 32 == 0, Co <= 256");
    DcnOutputs m;
    for (int k = 0; k < 8; ++k) m.ptr[k] = k < n_outputs ? outputs[k] : nullptr;
    m.n = n_outputs;
    m.group = dst_group;
    m.stride = dst_stride;
    m.offset = dst_offset;
    m.slab_rows = slab_rows;
    return dcn_forward_tc_impl(input, weight, with_bias ? bias : nullptr, conv_out, nullptr,
                               reinterpret_cast<const long long*>(max_idx), flow_scale, nullptr, s, workspace,
                               workspace_bytes, static_cast<cudaStream_t>(stream), layout_flags, out_slope, &m);
}

int mrefsr_dynagg_dcn_backward(const float* input, const float* weight, const float* conv_out, const int64_t* max_idx,
                               int flow_scale, const float* grad_output, float* grad_input, float* grad_weight,
                               float* grad_bias, float* grad_conv_out, int B, int C, int H, int W, int Co,
                               int deformable_group, int with_bias, int layout_flags, int mode, void* workspace,
                               size_t workspace_bytes, void* stream) {
    MREFSR_CHECK(input && weight && conv_out && max_idx && grad_output, ERR_BAD_ARG, "dynagg backward: null pointer argument");
    MREFSR_CHECK(!with_bias || grad_bias, ERR_BAD_ARG, "dynagg backward: with_bias set but grad_bias is NULL");
    MREFSR_CHECK((layout_flags & ~MREFSR_DCN_IN_NHWC) == 0, ERR_BAD_ARG, "dynagg backward: unknown layout flags 0x%x",
                 layout_flags);
    const int m = mode == MREFSR_DCN_AUTO ? MREFSR_DCN_TF32 : mode;
    MREFSR_CHECK(m != MREFSR_DCN_FP32, ERR_UNSUPPORTED,
                 "dynagg backward: the fused forward runs tf32 or tf32x3, so must its backward (mode fp32 refused)");
    MREFSR_CHECK(m == MREFSR_DCN_TF32 || m == MREFSR_DCN_TF32X3, ERR_BAD_ARG, "dynagg backward: unknown mode %d", mode);
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, 3, 3, 1, 1, 1, 1, 1, 1, 1, deformable_group);
    if (rc) return rc;
    // the fused forward's shapes; Co * positions < 2^31 keeps the coordinate gradients on the NHWC kernels
    MREFSR_CHECK(dcn_tc_eligible(s) && (size_t)B * Co * H * W < ((size_t)1 << 31), ERR_UNSUPPORTED,
                 "dynagg backward: needs C %% 32 == 0, (C/deformable_group) %% 8 == 0, Co %% 32 == 0, Co <= 256");
    MREFSR_CHECK(flow_scale >= 1 && H % flow_scale == 0 && W % flow_scale == 0, ERR_BAD_ARG,
                 "dynagg backward: output %dx%d not a multiple of the flow scale %d", H, W, flow_scale);
    DynAggSrc src;
    src.max_idx = reinterpret_cast<const long long*>(max_idx);
    src.flow_scale = flow_scale;
    src.hp = H / flow_scale - 2;
    src.wp = W / flow_scale - 2;
    src.x_nhwc = (layout_flags & MREFSR_DCN_IN_NHWC) ? 1 : 0;
    MREFSR_CHECK(src.hp > 0 && src.wp > 1, ERR_BAD_ARG, "dynagg backward: feature grid too small");
    MREFSR_CHECK(!src.x_nhwc || (reinterpret_cast<uintptr_t>(input) & 31) == 0, ERR_BAD_ARG,
                 "dynagg backward: NHWC input must be 32-byte aligned");
    return dcn_backward(input, weight, conv_out, nullptr, grad_output, grad_input, grad_weight, grad_bias, grad_conv_out,
                        nullptr, s, with_bias, m, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), src);
}

int mrefsr_dynagg_offsets(const float* conv_out,const float* pre_offset, float* offset, float* mask, float* abs_sum,
                          int B, int dg, int K, int H, int W, void* stream) {
    MREFSR_CHECK(conv_out && pre_offset && offset && mask && B > 0 && dg > 0 && K > 0 && H > 0 && W > 0, ERR_BAD_ARG,
                 "dynagg_offsets: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t total = (size_t)B * 3 * dg * K * H * W;
    ScopedTiming tm(MREFSR_K_GLUE, st);
    const int P = H * W;
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (P % 4 == 0 && al16(conv_out) && al16(pre_offset) && al16(offset) && al16(mask) && (size_t)B * 3 * dg * K <= 65535) {
        int gx = cdiv(P / 4, 256 * 2);
        if (gx > 4) gx = 4;
        if (gx < 1) gx = 1;
        dynagg_offsets_vec4_kernel<<<dim3(gx, B * 3 * dg * K), 256, 0, st>>>(conv_out, pre_offset, offset, mask, abs_sum, dg, K, P);
    } else {
        dynagg_offsets_kernel<<<grid_for(total), 256, 0, st>>>(conv_out, pre_offset, offset, mask, abs_sum, B, dg, K, P);
    }
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

int mrefsr_dynagg_offsets_backward(const float* grad_offset, const float* grad_mask, const float* mask, float* grad_conv_out,
                                   int B, int dg, int K, int H, int W, void* stream) {
    MREFSR_CHECK(grad_offset && grad_mask && mask && grad_conv_out && B > 0 && dg > 0 && K > 0 && H > 0 && W > 0, ERR_BAD_ARG,
                 "dynagg_offsets_backward: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t total = (size_t)B * 3 * dg * K * H * W;
    ScopedTiming tm(MREFSR_K_GLUE, st);
    const int P = H * W;
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (P % 4 == 0 && al16(grad_offset) && al16(grad_mask) && al16(mask) && al16(grad_conv_out) &&
        (size_t)B * 3 * dg * K <= 65535) {
        int gx = cdiv(P / 4, 256);
        if (gx > 8) gx = 8;
        dynagg_offsets_bwd_vec4_kernel<<<dim3(gx, B * 3 * dg * K), 256, 0, st>>>(grad_offset, grad_mask, mask, grad_conv_out, dg,
                                                                                  K, P);
    } else {
        dynagg_offsets_bwd_kernel<<<grid_for(total), 256, 0, st>>>(grad_offset, grad_mask, mask, grad_conv_out, B, dg, K, P);
    }
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

int mrefsr_modulated_deform_conv_forward_host(const float* input, const float* weight, const float* bias,
                                              const float* offset, const float* mask, float* output, int B, int C,
                                              int H, int W, int Co, int kh, int kw, int stride_h, int stride_w,
                                              int pad_h, int pad_w, int dil_h, int dil_w, int group,
                                              int deformable_group, int with_bias, int mode, void* stream) {
    DcnShape s;
    int rc = dcn_make_shape(&s, B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, group,
                            deformable_group);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int K = kh * kw, P = s.Ho * s.Wo;
    const size_t ws = align_up(mrefsr_dcn_workspace_bytes(B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w,
                                                          dil_h, dil_w, group, deformable_group, mode, 0), 1024);
    const size_t n_in = (size_t)B * C * H * W, n_w = (size_t)Co * (C / group) * K, n_off = (size_t)B * 2 * deformable_group * K * P,
                 n_mask = n_off / 2, n_out = (size_t)B * Co * P;
    size_t o = ws;
    auto take = [&](size_t elems) { size_t r = o; o += align_up(elems * 4, 1024); return r; };
    const size_t o_in = take(n_in), o_w = take(n_w), o_b = take(Co), o_off = take(n_off), o_mask = take(n_mask), o_out = take(n_out);
    void* base = nullptr;
    rc = arena_get(o, &base);
    if (rc) return rc;
    uint8_t* p = static_cast<uint8_t*>(base);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(p + off); };
    MREFSR_CUDA(cudaMemcpyAsync(F(o_in), input, n_in * 4, cudaMemcpyHostToDevice, st));
    MREFSR_CUDA(cudaMemcpyAsync(F(o_w), weight, n_w * 4, cudaMemcpyHostToDevice, st));
    if (with_bias) MREFSR_CUDA(cudaMemcpyAsync(F(o_b), bias, (size_t)Co * 4, cudaMemcpyHostToDevice, st));
    MREFSR_CUDA(cudaMemcpyAsync(F(o_off), offset, n_off * 4, cudaMemcpyHostToDevice, st));
    MREFSR_CUDA(cudaMemcpyAsync(F(o_mask), mask, n_mask * 4, cudaMemcpyHostToDevice, st));
    rc = mrefsr_modulated_deform_conv_forward(F(o_in), F(o_w), with_bias ? F(o_b) : nullptr, F(o_off), F(o_mask), F(o_out),
                                              B, C, H, W, Co, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, group,
                                              deformable_group, with_bias, mode, p, ws, st);
    if (rc) return rc;
    MREFSR_CUDA(cudaMemcpyAsync(output, F(o_out), n_out * 4, cudaMemcpyDeviceToHost, st));
    MREFSR_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // extern "C"
