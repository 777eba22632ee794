// mrefsr_b200/csrc/dcn_common.cuh -- shapes and the sampling rule shared by the DCN kernels.
#pragma once
#include "common.cuh"

namespace mrefsr {

struct DcnShape {
    int B, C, H, W, Co, kh, kw, sh, sw, ph, pw, dh, dw, G, DG, Ho, Wo;
};

__host__ __device__ __forceinline__ int cdiv_d(int a, int b) { return (a + b - 1) / b; }

// Sample sources of the DCN backward kernels: the type of their last argument selects the overload (dcn.cu).
// PlaneSrc: materialised offset [B, 2*DG*K, Ho, Wo] and mask [B, DG*K, Ho, Wo] planes (the kernels' offset / mask
// arguments); grad_offset / grad_mask are written as such planes.
struct PlaneSrc {};
// DynAggSrc: the fused DynAgg forward's inputs.  The kernels' `offset` argument is the raw conv_offset_mask output
// [B, 3*DG*K, Ho, Wo] (dy / dx of (g, k) in channels 2(g*K+k) / +1, mask logits in 2*DG*K + g*K + k), flows come from
// the matcher's arg-max map max_idx [B, hp, wp] at 1/flow_scale resolution, and the gradient with respect to that raw
// output is written in its layout (`grad_offset` argument).  x_nhwc: the input (and grad_input) is [B, H, W, C].
struct DynAggSrc {
    const long long* max_idx;
    int flow_scale, hp, wp, x_nhwc;
};

#ifdef __CUDACC__
// Bilinear sample of one channel plane at fractional (y, x).
// Rule of deform_conv_cuda_kernel.cu:618 + :468-497: the value is 0 unless -1 < y < H and -1 < x < W; inside,
// corners that fall outside the plane contribute 0.
__device__ __forceinline__ float dcn_sample(const float* __restrict__ plane, int H, int W, float y, float x) {
    if (!(y > -1.f && x > -1.f && y < (float)H && x < (float)W)) return 0.f;
    const int y0 = (int)floorf(y), x0 = (int)floorf(x);
    const int y1 = y0 + 1, x1 = x0 + 1;
    const float ly = y - (float)y0, lx = x - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const float a = (y0 >= 0 && x0 >= 0) ? __ldg(plane + y0 * W + x0) : 0.f;
    const float b = (y0 >= 0 && x1 <= W - 1) ? __ldg(plane + y0 * W + x1) : 0.f;
    const float c = (y1 <= H - 1 && x0 >= 0) ? __ldg(plane + y1 * W + x0) : 0.f;
    const float d = (y1 <= H - 1 && x1 <= W - 1) ? __ldg(plane + y1 * W + x1) : 0.f;
    return hy * hx * a + hy * lx * b + ly * hx * c + ly * lx * d;
}
#endif

int dcn_make_shape(DcnShape* s, int B, int C, int H, int W, int Co, int kh, int kw, int sh, int sw, int ph, int pw,
                   int dh, int dw, int G, int DG);
int dcn_forward_fp32(const float* x, const float* w, const float* bias, const float* off, const float* mask, float* out,
                     const DcnShape& s, cudaStream_t st);

// NCHW -> NHWC copy (dcn_tc.cu), also used by the backward's position-major im2col
// (xt_lo: the 3-pass split, xt = tf32(x) and xt_lo = tf32(x - xt))
int dcn_nchw_to_nhwc(const float* x, float* xt, int B, int C, int HW, cudaStream_t st, bool round_tf32 = false,
                     float* xt_lo = nullptr);

// tcgen05 TF32 GEMM D = A . B^T of the backward pass (gemm_tc.cu); A_lo / B_lo non-NULL: the 3-pass variant
// D = A_lo . B^T + A . B_lo^T + A . B^T (A, B then hold the hi planes; the lo planes share their pitches and strides)
bool gemm_tc_operands_ok(const void* A, int lda, long long a_batch_stride, const void* B, int ldb, long long b_batch_stride);
int gemm_tf32_nt(const float* A, int lda, long long a_batch_stride, const float* B, int ldb, long long b_batch_stride,
                 float* D, int ldd, long long d_stride, int M, int N, int K, int batch, int reduce, int splits,
                 cudaStream_t st, const float* A_lo = nullptr, const float* B_lo = nullptr);

int dcn_pack_weights(const float* w, float* wt, int Co, int C, int K, cudaStream_t st, bool x3 = false);

// several destination buffers for one forward (reference-sharded mode: local + peer copies of the gathered tensor)
struct DcnOutputs {
    float* ptr[8];
    int n, group, stride, offset;   // sample b -> slot (b / group) * stride + offset + b % group  (group 0: slot b)
    int slab_rows;                  // > 0: output row oy goes to buffer oy / slab_rows only ([slots, Co, slab_rows, Wo])
};

// tcgen05 (TF32) forward, dcn_tc.cu
bool dcn_tc_eligible(const DcnShape& s);
size_t dcn_tc_workspace_bytes(const DcnShape& s, int mode);
int dcn_forward_tc_impl(const float* x, const float* w, const float* bias, const float* off, const float* mask,
                        const long long* max_idx, int flow_scale, float* out, const DcnShape& s, void* workspace,
                        size_t workspace_bytes, cudaStream_t st, int layout_flags, float out_slope,
                        const DcnOutputs* multi);
int dcn_tc_tile_plan(int B, int Ho, int Wo, int* meta, int* coords, size_t max_rows);
int dcn_forward_tc(const float* x, const float* w, const float* bias, const float* off, const float* mask, float* out,
                   const DcnShape& s, void* workspace, size_t workspace_bytes, cudaStream_t st, bool x3);

}  // namespace mrefsr
