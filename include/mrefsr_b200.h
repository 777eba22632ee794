/*
 * mrefsr_b200.h -- C ABI of libmrefsr_b200.so: the B200-native (sm_100a) implementation of
 * MRefSR's reference-alignment hot path.
 *
 * Boundary rules
 *   - extern "C", plain pointers and sizes only; no torch / ATen types.
 *   - All tensor pointers are DEVICE pointers to contiguous row-major (NCHW) buffers unless the
 *     function name ends in _host.  `stream` is a cudaStream_t passed as void* (NULL = default
 *     stream).  Calls are asynchronous with respect to the host, like the reference's kernels
 *     (basicsr/ops/dcn/src/deform_conv_cuda_kernel.cu:788 launches on the current stream).
 *   - The caller owns every buffer, including the scratch `workspace` whose size the matching
 *     *_workspace_bytes() function reports (the reference's `ones` / `columns` scratch tensors,
 *     basicsr/ops/dcn/deform_conv.py:148, play the same role).
 *   - Return value: 0 on success, negative on error; mrefsr_last_error() returns the message of
 *     the last failing call on this thread.  There is no CPU fallback anywhere: a missing GPU or
 *     an unsupported configuration is an error, never a silent slow path.
 *
 * Each entry point cites the reference interface (file:line under /root/reference) it replaces.
 */
#ifndef MREFSR_B200_H_
#define MREFSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MREFSR_ABI_VERSION 1

#if defined(__GNUC__)
#define MREFSR_API __attribute__((visibility("default")))
#else
#define MREFSR_API
#endif

MREFSR_API int mrefsr_abi_version(void);
MREFSR_API const char* mrefsr_last_error(void);
/* number of SMs of the current device (148 on B200); negative on error */
MREFSR_API int mrefsr_sm_count(void);

/* ------------------------------------------------------------------------------------------
 * (1) Correspondence matcher
 *     replaces  basicsr/archs/ref_map_util.py:26-86  feature_match_index(feat_input, feat_ref,
 *               patch_size, input_stride, ref_stride, is_norm, norm_input)
 *     batched over the (image, reference) pairs that basicsr/archs/corres_generation_arch.py:53
 *     and basicsr/models/multi_ref_restoration_model.py:287 loop over in Python.
 *
 * feat_in  [n_in,  C, h_in,  w_in ]  fp32     feat_ref [n_pairs, C, h_ref, w_ref] fp32
 * pair p is matched against input  (p / in_div) % n_in   (pairs laid out [B,R]: in_div = R;
 * laid out [R,B]: in_div = 1).
 * normalize_pixels != 0 first applies F.normalize(x.reshape(C,-1), dim=0) (eps 1e-12) to both,
 * i.e. corres_generation_arch.py:57-59.
 * max_idx [n_pairs, h', w'] int64 (value y_ref * w'_ref + x_ref), max_val [n_pairs, h', w'] fp32,
 * h' = (h_in - patch_size) / input_stride + 1 etc.  Ties resolve to the lowest reference index
 * (torch.max semantics, ref_map_util.py:69-76).
 *
 * mode: MREFSR_MATCH_AUTO picks the tcgen05 path when patch_size == 3, both strides == 1 and
 *       C % 64 == 0, else the fp32 CUDA-core path.
 *       MREFSR_MATCH_TC_BF16X3: tcgen05 with 3-pass split-bf16 operands (fp32-grade similarities);
 *       MREFSR_MATCH_TC_BF16:   tcgen05 single bf16 pass (fast, similarity error ~1e-4);
 *       MREFSR_MATCH_FP32:      exact-fp32 CUDA-core kernel, any patch_size / stride.
 * ------------------------------------------------------------------------------------------ */
enum {
    MREFSR_MATCH_AUTO = 0,
    MREFSR_MATCH_TC_BF16X3 = 1,
    MREFSR_MATCH_TC_BF16 = 2,
    MREFSR_MATCH_FP32 = 3,
};
/* tuning flags OR-ed into `mode` (bits 8..): see DESIGN.md "matcher kernel" */
#define MREFSR_MATCH_FLAG_NO_STRIP 0x100      /* one tap per pipeline stage (no row-shifted descriptors) */
#define MREFSR_MATCH_FLAG_BASE_OFFSET 0x200   /* encode (addr>>7)&7 in the descriptor base-offset field */
#define MREFSR_MATCH_FLAG_NO_DIAG 0x400       /* all nine taps as MMAs (round-1 kernel) instead of the diagonal form */
#define MREFSR_MATCH_FLAG_NO_BSTRIP 0x800     /* diagonal form: reload the reference rows per tap row (no shared strip) */

/* Introspection of the matcher's kernel choice and tiling for one pair (host logic only, no GPU work; tests/test_abi.py):
 * meta[0] kernel: 0 CUDA-core fp32, 1 nine-tap one tap per stage, 2 nine-tap strip, 3 diagonal form, 4 diagonal form with
 * the B strip;  meta[1], meta[2] M / N tiles;  meta[3], meta[4] output rows / columns owned by a tile;  meta[5], meta[6]
 * pixel-linear rows of the input / reference grids that are computed (tensor-core kernels);  meta[7] pipeline stages;
 * meta[8] dynamic shared memory in bytes;  meta[9] resolved mode.  meta must hold 10 ints. */
MREFSR_API int mrefsr_match_plan(int C, int h_in, int w_in, int h_ref, int w_ref, int patch_size, int input_stride,
                      int ref_stride, int mode, int* meta);
MREFSR_API size_t mrefsr_match_workspace_bytes(int n_in, int n_pairs, int C, int h_in, int w_in, int h_ref, int w_ref,
                                    int mode);
MREFSR_API int mrefsr_feature_match_batched(const float* feat_in, const float* feat_ref, int n_in, int n_pairs, int in_div,
                                 int C, int h_in, int w_in, int h_ref, int w_ref, int patch_size, int input_stride,
                                 int ref_stride, int is_norm, int norm_input, int normalize_pixels, int mode,
                                 int64_t* max_idx, float* max_val, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* idx -> flow -> nine zero-filled shifts at three scales.
 *     replaces  basicsr/archs/corres_generation_arch.py:30-47 (index_to_flow) and :70-105,
 *               basicsr/archs/arch_util.py:386-410 (tensor_shift)
 * max_idx [n, h-2, w-2] int64  ->  out_s1 [n,9,h,w,2], out_s2 [n,9,2h,2w,2], out_s4 [n,9,4h,4w,2]
 * fp32, last dim (x, y).  Any of the outputs may be NULL. */
MREFSR_API int mrefsr_pre_offsets(const int64_t* max_idx, int n, int h, int w, float* out_s1, float* out_s2, float* out_s4,
                       void* stream);

/* ------------------------------------------------------------------------------------------
 * (2) Modulated deformable convolution (DCNv2)
 *     replaces  basicsr/ops/dcn/src/deform_conv_ext.cpp:107-147 (pybind exports
 *               modulated_deform_conv_forward / modulated_deform_conv_backward) and the host code
 *               basicsr/ops/dcn/src/deform_conv_cuda.cpp:490-685.
 * input  [B, C, H, W]   weight [Co, C/group, kh, kw]   bias [Co] or NULL (with_bias = 0)
 * offset [B, 2*dg*kh*kw, Ho, Wo]  (channel 2*(g*K+k) = dy, +1 = dx)   mask [B, dg*kh*kw, Ho, Wo]
 * output [B, Co, Ho, Wo], overwritten.  The reference's `ones` / `columns` scratch tensors are
 * replaced by `workspace`.
 * mask == NULL means an all-ones mask: with bias == NULL that is DCNv1 (deform_conv_forward,
 * deform_conv_ext.cpp:52-66; same sampling rule, deform_conv_cuda_kernel.cu:84-112, 190-243).
 * mode: MREFSR_DCN_AUTO / MREFSR_DCN_FP32 (CUDA-core, exact fp32) / MREFSR_DCN_TF32 (tcgen05) /
 *       MREFSR_DCN_TF32X3 (tcgen05 with 3-pass split-tf32 operands, hi.hi + hi.lo + lo.hi: fp32-grade results, same
 *       shapes as MREFSR_DCN_TF32; in the backward it applies to the two GEMMs that MREFSR_DCN_TF32 runs on tcgen05).
 * ------------------------------------------------------------------------------------------ */
enum {
    MREFSR_DCN_AUTO = 0,
    MREFSR_DCN_FP32 = 1,
    MREFSR_DCN_TF32 = 2,
    MREFSR_DCN_TF32X3 = 3,
};
/* backward = 0: the scratch of the forward entry points; backward = 1: that of mrefsr_modulated_deform_conv_backward and
 * of mrefsr_dynagg_dcn_backward (called with 3x3, stride 1, pad 1, dil 1, group 1 and the mode passed to it). */
MREFSR_API size_t mrefsr_dcn_workspace_bytes(int B, int C, int H, int W, int Co, int kh, int kw, int stride_h, int stride_w,
                                  int pad_h, int pad_w, int dil_h, int dil_w, int group, int deformable_group,
                                  int mode, int backward);
/* Host-only introspection of the tcgen05 DCN kernel's work decomposition (no device work; used by the CPU tests):
 * how the B*Ho*Wo output positions of a call are laid out over 256-row CTA tiles.  meta[4] = {patches (1) or
 * consecutive positions (0), patch width, patch height, number of tiles}; coords (optional, 3 ints per row, room for
 * max_rows rows) receives (sample, oy, ox) of every row of every tile, (-1, -1, -1) for padding rows. */
MREFSR_API int mrefsr_dcn_tile_plan(int B, int Ho, int Wo, int* meta, int* coords, size_t max_rows);
MREFSR_API int mrefsr_modulated_deform_conv_forward(const float* input, const float* weight, const float* bias,
                                         const float* offset, const float* mask, float* output, int B, int C, int H,
                                         int W, int Co, int kh, int kw, int stride_h, int stride_w, int pad_h,
                                         int pad_w, int dil_h, int dil_w, int group, int deformable_group,
                                         int with_bias, int mode, void* workspace, size_t workspace_bytes,
                                         void* stream);
/* grad_input / grad_offset / grad_mask are overwritten; grad_weight / grad_bias are ACCUMULATED
 * into (the reference accumulates with addmm_ beta = 1 into caller-zeroed tensors,
 * deform_conv_cuda.cpp:659-671).  grad_input, grad_weight, grad_offset (+ grad_mask) may each be NULL (that
 * part is skipped); mask == NULL = all-ones mask, which gives DCNv1's deform_conv_backward_input /
 * deform_conv_backward_parameters (deform_conv_ext.cpp:68-105). */
MREFSR_API int mrefsr_modulated_deform_conv_backward(const float* input, const float* weight, const float* offset,
                                          const float* mask, const float* grad_output, float* grad_input,
                                          float* grad_weight, float* grad_bias, float* grad_offset, float* grad_mask,
                                          int B, int C, int H, int W, int Co, int kh, int kw, int stride_h,
                                          int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int group,
                                          int deformable_group, int with_bias, int mode, void* workspace,
                                          size_t workspace_bytes, void* stream);

/* DynAgg glue, fused: conv_out [B, 3*dg*9, H, W] (raw conv_offset_mask output) + pre_offset
 * [B, 9, H, W, 2] (x, y)  ->  offset [B, 2*dg*9, H, W], mask [B, dg*9, H, W] (sigmoid), and the
 * mean |learned offset| accumulated into *abs_sum (device float, may be NULL) instead of the
 * reference's host sync.
 *     replaces  basicsr/archs/ref_mrapa_restoration_arch.py:55-73 */
MREFSR_API int mrefsr_dynagg_offsets(const float* conv_out, const float* pre_offset, float* offset, float* mask,
                          float* abs_sum, int B, int dg, int K, int H, int W, void* stream);
/* Its backward (training): grad_conv_out [B, 3*dg*K, H, W] = [grad_offset, grad_mask * mask * (1 - mask)]
 * (the autograd of the chunk / cat / sigmoid sequence at ref_mrapa_restoration_arch.py:55-68; the pre-offsets carry no
 * gradient), one pass. */
MREFSR_API int mrefsr_dynagg_offsets_backward(const float* grad_offset, const float* grad_mask, const float* mask,
                                   float* grad_conv_out, int B, int dg, int K, int H, int W, void* stream);

/* Fused DynAgg forward: DCNv2 whose offsets / masks are assembled inside the gather from the raw conv_offset_mask
 * output and the matcher's arg-max map, so neither the pre-offset tensors nor offset / mask are ever written to HBM
 * (inference; for training, mrefsr_dynagg_dcn_backward below is its backward from the same source):
 *   offset[:, 2(g*9+k)  ] = conv_out[:, 2(g*9+k)  ] + s * flow_y[Y/s - i, X/s - j]      (k = 3i + j)
 *   offset[:, 2(g*9+k)+1] = conv_out[:, 2(g*9+k)+1] + s * flow_x[Y/s - i, X/s - j]
 *   mask = sigmoid(conv_out[:, 2*dg*9 + g*9 + k]),  flow = index_to_flow(max_idx) (0 outside the grid)
 *     replaces  basicsr/archs/ref_mrapa_restoration_arch.py:45-76 (DynAgg.forward) together with
 *               basicsr/archs/corres_generation_arch.py:30-47, :70-105 for one scale.
 * input [B,C,H,W], conv_out [B,3*dg*9,H,W], max_idx [B,H/s-2,W/s-2] int64, 3x3 kernel, stride 1, pad 1, dil 1.
 * Requires the tcgen05 path (C % 32 == 0, (C/dg) % 4 == 0, Co % 32 == 0, Co <= 256). */
MREFSR_API int mrefsr_dynagg_dcn_forward(const float* input, const float* weight, const float* bias, const float* conv_out,
                              const int64_t* max_idx, int flow_scale, float* output, int B, int C, int H, int W,
                              int Co, int deformable_group, int with_bias, void* workspace, size_t workspace_bytes,
                              void* stream);
/* Same, for a channels-last caller (SURVEY 8f-3, feature hand-off layout): layout_flags says that `input` already
 * is [B, H, W, C] (the layout the gather wants: no transpose pass) and / or that `output` is to be written as
 * [B, H, W, Co]; conv_out stays [B, 3*dg*9, H, W] planes.  out_slope: leaky-ReLU slope applied to the output in the
 * epilogue (the lrelu that follows DynAgg at ref_mrapa_restoration_arch.py:228-229; 1.0f = none). */
enum {
    MREFSR_DCN_IN_NHWC = 1,
    MREFSR_DCN_OUT_NHWC = 2,
    MREFSR_DCN_W_PACKED = 4, /* `weight` is the output of mrefsr_dcn_pack_weights (inference: packed once per weight update) */
    MREFSR_DCN_X3 = 8,       /* 3-pass split-tf32 operands (as mode MREFSR_DCN_TF32X3); with MREFSR_DCN_W_PACKED the
                                weight must come from mrefsr_dcn_pack_weights_x3; workspace: mrefsr_dcn_workspace_bytes
                                with mode MREFSR_DCN_TF32X3 */
};
/* The plain GEMM of the DCN backward on tcgen05 (csrc/gemm_tc.cu; TF32 operands, fp32 accumulate), exported for tests:
 *   D[m][n] = sum_k A[m][k] * B[n][k],   A [M x K] and B [N x K] row-major (k contiguous), D row-major with pitch ldd.
 * reduce == 0: `batch` independent products, operands / outputs a_batch_stride / b_batch_stride / d_stride elements
 *   apart (a_batch_stride == 0: one A for all) -- columns = W^T . grad_output, deform_conv_cuda.cpp:623-626;
 * reduce != 0: ONE product summed over the batch as well as over k, computed as `splits` partial sums written to
 *   D + split * d_stride (the caller adds them in split order: deterministic) -- grad_weight += grad_output .
 *   columns^T, deform_conv_cuda.cpp:659-664.
 * Pitches and batch strides must be multiples of 4 floats and the bases 16-byte aligned (TMA). */
MREFSR_API int mrefsr_gemm_tf32_nt(const float* A, int lda, long long a_batch_stride, const float* B, int ldb,
                                   long long b_batch_stride, float* D, int ldd, long long d_stride, int M, int N, int K,
                                   int batch, int reduce, int splits, void* stream);
/* The same GEMM with 3-pass split-tf32 operands (the backward of mode MREFSR_DCN_TF32X3): each operand comes as a tf32 hi
 * plane and a tf32 lo plane (x = hi + lo, both with the same pitch and batch stride), and
 *   D = A_lo . B_hi^T + A_hi . B_lo^T + A_hi . B_hi^T   accumulated in fp32 (fp32-grade products; A_lo . B_lo^T is dropped). */
MREFSR_API int mrefsr_gemm_tf32x3_nt(const float* A_hi, const float* A_lo, int lda, long long a_batch_stride,
                                     const float* B_hi, const float* B_lo, int ldb, long long b_batch_stride, float* D,
                                     int ldd, long long d_stride, int M, int N, int K, int batch, int reduce, int splits,
                                     void* stream);
/* W[Co][C][kh*kw] (the reference's parameter layout, deform_conv.py:305-309) -> the tcgen05 kernels' B operand
 * [Co][tap][C], rounded to tf32 (round to nearest, so the tensor core's truncation is exact).  The forward entry
 * points do this on every call unless MREFSR_DCN_W_PACKED is set; a module whose weights are frozen packs once. */
MREFSR_API int mrefsr_dcn_pack_weights(const float* weight, float* packed, int Co, int C, int K, void* stream);
/* The B operand of the 3-pass kernels (MREFSR_DCN_X3): [Co][tap][C/16][hi c0..7 | hi c8..15 | lo c0..7 | lo c8..15],
 * 2*K*C floats per output channel, hi = tf32(w), lo = tf32(w - hi).  C % 16 == 0. */
MREFSR_API int mrefsr_dcn_pack_weights_x3(const float* weight, float* packed, int Co, int C, int K, void* stream);
MREFSR_API int mrefsr_dynagg_dcn_forward_ex(const float* input, const float* weight, const float* bias,
                                 const float* conv_out, const int64_t* max_idx, int flow_scale, float* output, int B,
                                 int C, int H, int W, int Co, int deformable_group, int with_bias, int layout_flags,
                                 float out_slope, void* workspace, size_t workspace_bytes, void* stream);
/* Same, with the exchange step of the reference-sharded mode (SURVEY 8e, config 4) folded into the epilogue: every
 * finished output tile is stored to each of `outputs[0..n_outputs)` -- this GPU's and the peers' copies of the
 * gathered tensor [n, R, Co, H, W], peer copies being NVLink-mapped device pointers (CUDA IPC / symmetric memory) --
 * at sample slot (b / dst_group) * dst_stride + dst_offset + b % dst_group (dst_group = references held by this rank,
 * dst_stride = R, dst_offset = first global reference of this rank; dst_group = 0: slot b).  Replaces
 * {DCN -> transpose copy -> ncclAllGather -> cat}; the caller still needs a cross-GPU barrier before the consumer
 * reads the buffer and before the next forward overwrites it.  `outputs` is a HOST array of device pointers. */
MREFSR_API int mrefsr_dynagg_dcn_forward_multi(const float* input, const float* weight, const float* bias,
                                    const float* conv_out, const int64_t* max_idx, int flow_scale,
                                    float* const* outputs, int n_outputs, int dst_group, int dst_stride,
                                    int dst_offset, int B, int C, int H, int W, int Co, int deformable_group,
                                    int with_bias, int layout_flags, float out_slope, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* Same with PIXEL-SLAB routing: output row oy is stored to outputs[oy / slab_rows] only (buffers in RANK order, each
 * [n, R, Co, slab_rows, W] NCHW planes, slot as above).  Each rank of the reference-sharded mode then holds every
 * reference's aligned features for ITS rows, runs the fusion (softmax over references,
 * ref_mrapa_restoration_arch.py:321-335) on 1/N of the pixels and all-gathers the fused result: the exchange of SURVEY
 * 8e as an all-to-all inside the DCN epilogue, N times fewer bytes per GPU than the all-gather of aligned features. */
MREFSR_API int mrefsr_dynagg_dcn_forward_slabs(const float* input, const float* weight, const float* bias,
                                    const float* conv_out, const int64_t* max_idx, int flow_scale,
                                    float* const* outputs, int n_outputs, int slab_rows, int dst_group, int dst_stride,
                                    int dst_offset, int B, int C, int H, int W, int Co, int deformable_group,
                                    int with_bias, int layout_flags, float out_slope, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* Backward of the fused DynAgg forward (training): the gradients of mrefsr_dynagg_dcn_forward_ex's output with respect
 * to input, weight, bias and the raw conv_offset_mask output, read from the same conv_out + max_idx source.  The
 * sampling points and masks are computed bit for bit as the forward computes them, and no offset / mask / pre-offset
 * tensor is materialised:
 *   grad_conv_out[:, 2(g*9+k)], [:, 2(g*9+k)+1] = d loss / d offset (y, x)   (the flows carry no gradient)
 *   grad_conv_out[:, 2*dg*9 + g*9 + k]          = d loss / d mask * mask * (1 - mask)
 * Shapes and requirements as mrefsr_dynagg_dcn_forward (3x3, stride 1, pad 1, dil 1, the tcgen05 shapes, H and W
 * multiples of flow_scale); grad_output [B, Co, H, W] planes, grad_conv_out [B, 3*dg*9, H, W] planes (overwritten).
 * grad_input, grad_weight and grad_conv_out may each be NULL (that part is skipped); grad_input is overwritten, in
 * input's layout; grad_weight / grad_bias are ACCUMULATED into, as in mrefsr_modulated_deform_conv_backward.
 * layout_flags: MREFSR_DCN_IN_NHWC (input and grad_input are [B, H, W, C]; input 32-byte aligned) or 0.
 * mode: MREFSR_DCN_TF32 (MREFSR_DCN_AUTO resolves to it) or MREFSR_DCN_TF32X3, the modes the fused forward runs;
 * MREFSR_DCN_FP32 is refused with ERR_UNSUPPORTED.  workspace: mrefsr_dcn_workspace_bytes(B, C, H, W, Co, 3, 3, 1, 1,
 * 1, 1, 1, 1, 1, deformable_group, mode, 1), the size of the materialised backward. */
MREFSR_API int mrefsr_dynagg_dcn_backward(const float* input, const float* weight, const float* conv_out,
                                          const int64_t* max_idx, int flow_scale, const float* grad_output,
                                          float* grad_input, float* grad_weight, float* grad_bias, float* grad_conv_out,
                                          int B, int C, int H, int W, int Co, int deformable_group, int with_bias,
                                          int layout_flags, int mode, void* workspace, size_t workspace_bytes,
                                          void* stream);

/* ------------------------------------------------------------------------------------------
 * Trunk glue (SURVEY 8f-2: the plain-convolution network either side of the path; convolutions
 * themselves stay cuDNN).  One streaming pass instead of torch's bias-add / activation /
 * residual-add kernels:
 *   mrefsr_bias_act:      x[b,c,:] = act(x[b,c,:] + bias[c]) * scale + residual[b,c,:]   (in place)
 *       ResidualBlockNoBN (basicsr/archs/arch_util.py:88-117), offset convs + tails
 *       (ref_mrapa_restoration_arch.py:140-259), VGG conv+ReLU (vgg_arch.py:141-161),
 *       MRAPAFusion embeddings conv+PReLU (* C^-0.5) (ref_mrapa_restoration_arch.py:293-302, 321-323).
 *       bias / residual may be NULL; slope_dev (device, 1 or C entries: nn.PReLU weight) overrides
 *       `slope` when non-NULL.  x, residual: dense fp32, NCHW planes (channels_last = 0) or NHWC
 *       (channels_last = 1, torch.channels_last), HW = H*W.
 *       res_div: sample b of x takes residual sample b / res_div (a per-image term shared by its res_div
 *       references; 1 = same batch).  res_pre = 1 adds the residual before the activation instead:
 *       x = act(x + bias + residual) * scale  -- the per-image half of a convolution over cat([x, feat]) that
 *       was split by input channels (small/medium/large_offset_conv1, ref_mrapa_restoration_arch.py:222-227).
 *   mrefsr_layout_convert: dense [B,C,HW] <-> [B,HW,C] (torch.channels_last), C % 4 == 0, out of place;
 *       bias (C entries, may be NULL) is added on the way: a convolution's bias folded into the conversion.
 *   mrefsr_attn_modulate: refs = refs * sigmoid(attn_mul + bias_mul[c]) * 2 + (attn_add + bias_add[c])
 *       (ref_mrapa_restoration_arch.py:341-344), in place on refs.
 * ------------------------------------------------------------------------------------------ */
enum {
    MREFSR_ACT_NONE = 0,
    MREFSR_ACT_LEAKY = 1,   /* v > 0 ? v : slope * v   (ReLU: slope 0; PReLU: slope_dev) */
    MREFSR_ACT_SIGMOID = 2,
};
MREFSR_API int mrefsr_bias_act(float* x, const float* bias, const float* slope_dev, int slope_n, const float* residual,
                    int res_div, int res_pre, int B, int C, int HW, int channels_last, int act, float slope,
                    float scale, void* stream);
MREFSR_API int mrefsr_layout_convert(const float* src, float* dst, const float* bias, int B, int C, int HW,
                          int to_channels_last, void* stream);
/* Training path of the same epilogue, channels-last activations [rows = B*H*W, C], dtype 0 = fp32 / 1 = bf16 (the
 * reference's training step runs these as separate torch kernels: bias add, activation, their backward, and a reduction
 * over grad_output for every convolution's bias gradient -- basicsr/archs/arch_util.py:88-117 under autograd).
 *   forward:  x = act(x + bias[c]) * scale + residual   in place (residual may be NULL; act NONE or LEAKY)
 *   backward: grad_in = grad_out * act'(y) * scale (y = the forward's output; only read for LEAKY, which then requires
 *             residual == NULL and scale > 0 in the forward), grad_bias[c] = sum over rows of grad_in, in one pass;
 *             grad_in may be NULL when only the bias gradient is wanted.  partial: fp32 scratch of
 *             mrefsr_bias_act_train_blocks() * C entries (partial sums are added in a fixed order: deterministic).
 *   mrefsr_bias_act_train_supported: 1 when C fits the 16-byte channel vectors of these kernels. */
MREFSR_API int mrefsr_bias_act_train_supported(int C, int dtype);
MREFSR_API int mrefsr_bias_act_train_blocks(void);
MREFSR_API int mrefsr_bias_act_train_forward(void* x, const float* bias, const void* residual, long long rows, int C,
                                  int dtype, int act, float slope, float scale, void* stream);
MREFSR_API int mrefsr_bias_act_train_backward(const void* grad_out, const void* y, void* grad_in, float* grad_bias,
                                   float* partial, long long rows, int C, int dtype, int act, float slope,
                                   float scale, void* stream);
/* The two conversions of the training path under bf16 autocast, one pass each (torch: a cast, then a strided copy):
 * to_channels_last_bf16 = 0: bf16 channels-last [B,HW,C] -> fp32 planes [B,C,HW];  1: fp32 planes -> bf16 channels-last
 * (round to nearest even).  C % 4 == 0. */
MREFSR_API int mrefsr_layout_convert_bf16(const void* src, void* dst, int B, int C, int HW, int to_channels_last_bf16,
                               void* stream);
/* The same with a leaky ReLU folded in (the activation after DynAgg, ref_mrapa_restoration_arch.py:229):
 * to_channels_last_bf16 = 1: dst = lrelu(src, slope) on the way out;  0: dst = src * (gate > 0 ? 1 : slope), gate = the
 * activation's bf16 channels-last OUTPUT (its backward on the way in; gate may be NULL). */
MREFSR_API int mrefsr_layout_convert_bf16_act(const void* src, void* dst, const void* gate, float slope, int B, int C, int HW,
                                   int to_channels_last_bf16, void* stream);
/* 2x2 / stride-2 max pooling, channels-last [B,H,W,C] -> [B,H/2,W/2,C] (VGG pool1 / pool2), C % 4 == 0, H, W even. */
MREFSR_API int mrefsr_maxpool2x2_nhwc(const float* src, float* dst, int B, int C, int H, int W, void* stream);
MREFSR_API int mrefsr_attn_modulate(float* refs, const float* attn_mul, const float* attn_add, const float* bias_mul,
                         const float* bias_add, int B, int C, int HW, int channels_last, void* stream);

/* ------------------------------------------------------------------------------------------
 * (3) Multi-reference attention fusion core
 *     replaces  basicsr/archs/ref_mrapa_restoration_arch.py:321-335
 * emb_t [n, C, h, w] (already scaled by C^-0.5), emb [n*t, C, h, w], ass [n*t, Cv, h, w]
 * out [n, Cv, h, w] = sum_t softmax_t(<emb_t, emb_t'>)[t] * ass[t];  prob [n, t, h, w] optional
 * (saved for backward; may be NULL).
 * ------------------------------------------------------------------------------------------ */
MREFSR_API int mrefsr_mrapa_attention_forward(const float* emb_t, const float* emb, const float* ass, float* out, float* prob,
                                   int n, int t, int C, int Cv, int h, int w, void* stream);
/* Channels-last inference variant with the producing convolutions' epilogues folded in: the inputs are the RAW
 * cuDNN outputs of conv_emb1 / conv_emb2 / conv_ass in NHWC ([n,h,w,C], [n*t,h,w,C], [n*t,h,w,Cv]);
 * q = prelu(q_raw + bias_q, slope_q) * q_scale, k = prelu(k_raw + bias_k, slope_k), v = v_raw + bias_v are applied
 * on the fly (ref_mrapa_restoration_arch.py:293-302, 321-323), out [n,h,w,Cv].  Any bias / slope pointer may be
 * NULL (no bias / no activation); slope_*_n is 1 or C (nn.PReLU).  C in {64,128,256}, Cv = 2C, t <= 8. */
MREFSR_API int mrefsr_mrapa_attention_nhwc(const float* q_raw, const float* k_raw, const float* v_raw, const float* bias_q,
                                const float* bias_k, const float* bias_v, const float* slope_q, int slope_q_n,
                                const float* slope_k, int slope_k_n, float q_scale, float* out, int n, int t, int C,
                                int Cv, int h, int w, void* stream);
/* bf16 tensors in and out (inference; the north star's "bf16 tolerance stated separately"): same kernel, half the bytes,
 * logits / softmax / weighted sum in fp32, output rounded to nearest even.  Tolerance against the fp64 oracle evaluated on
 * the SAME bf16-rounded inputs: 4e-3 of the output scale (one bf16 rounding of the result = 2^-9 relative).  Needs t <= 8,
 * h*w % 4 == 0, 8-byte aligned tensors. */
MREFSR_API int mrefsr_mrapa_attention_forward_bf16(const void* emb_t, const void* emb, const void* ass, void* out, int n,
                                                   int t, int C, int Cv, int h, int w, void* stream);
MREFSR_API int mrefsr_mrapa_attention_backward(const float* emb_t, const float* emb, const float* ass, const float* prob,
                                    const float* grad_out, float* grad_emb_t, float* grad_emb, float* grad_ass,
                                    int n, int t, int C, int Cv, int h, int w, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-buffer variants (end-to-end path): copy inputs host->device, run, copy results back, and
 * synchronise the stream before returning.  Device scratch comes from an internal arena that
 * grows on demand (mrefsr_arena_release() frees it).
 * ------------------------------------------------------------------------------------------ */
MREFSR_API int mrefsr_feature_match_batched_host(const float* feat_in, const float* feat_ref, int n_in, int n_pairs,
                                      int in_div, int C, int h_in, int w_in, int h_ref, int w_ref, int patch_size,
                                      int input_stride, int ref_stride, int is_norm, int norm_input,
                                      int normalize_pixels, int mode, int64_t* max_idx, float* max_val,
                                      void* stream);
MREFSR_API int mrefsr_modulated_deform_conv_forward_host(const float* input, const float* weight, const float* bias,
                                              const float* offset, const float* mask, float* output, int B, int C,
                                              int H, int W, int Co, int kh, int kw, int stride_h, int stride_w,
                                              int pad_h, int pad_w, int dil_h, int dil_w, int group,
                                              int deformable_group, int with_bias, int mode, void* stream);
MREFSR_API int mrefsr_mrapa_attention_forward_host(const float* emb_t, const float* emb, const float* ass, float* out, int n,
                                        int t, int C, int Cv, int h, int w, void* stream);
MREFSR_API void mrefsr_arena_release(void);

/* Per-kernel device timing for the roofline report (bench.py).  When enabled, the main kernel of each piece
 * is bracketed by CUDA events recorded on the launching stream; mrefsr_timing_read() synchronises those
 * events and returns the accumulated milliseconds and launch count per kernel id, then resets. */
enum {
    MREFSR_K_MATCH_MAIN = 0, /* correlation + arg-max kernel (tcgen05 or fp32) */
    MREFSR_K_MATCH_PREP = 1, /* layout / split / norms / finalize around it */
    MREFSR_K_DCN_FWD = 2,    /* DCN forward main kernel */
    MREFSR_K_DCN_AUX = 3,    /* DCN layout / weight repack kernels */
    MREFSR_K_FUSION_FWD = 4, /* attention core */
    MREFSR_K_GLUE = 5,       /* pre-offsets, DynAgg offset/mask assembly */
    MREFSR_K_COUNT = 6
};
MREFSR_API void mrefsr_timing_enable(int on);
MREFSR_API int mrefsr_timing_read(double* ms_out, unsigned long long* launches_out, int n);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
MREFSR_API unsigned long long mrefsr_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MREFSR_B200_H_ */
