// mrefsr_b200/csrc/gemm_tc.cu -- the two plain GEMMs of the DCN backward on tcgen05 (TF32 operands, fp32 accumulate).
//
// Replaces the addmm_ calls of basicsr/ops/dcn/src/deform_conv_cuda.cpp:623-626 (columns = W^T . grad_output) and
// :659-664 (grad_weight += grad_output . columns^T), which round 1 handed to cuBLAS.  One kernel serves both:
//
//     D[m][n] = sum_k A[m][k] * B[n][k]          A, B row-major with k contiguous ("NT"), D row-major
//
//   per-batch mode   : D[z] = A[z or shared] . B[z]^T for every batch item z (the columns GEMM: A = W^T shared,
//                      B = grad_output of sample z position-major, D = columns of sample z);
//   reduce mode      : one D summed over the batch as well as over k (the grad_weight GEMM: k = output positions,
//                      batch = samples), the flattened (z, k-block) range cut into `splits` contiguous pieces whose
//                      partial sums land in D[split] and are added up by the caller in a fixed order (deterministic).
//
// Persistent CTAs, 128 x 128 output tiles, K step 32 (128-byte rows, SWIZZLE_128B), both operands by TMA (rows / k
// beyond the matrix are zero-filled by the copy engine, so no tile needs padding in memory), 6-stage ring, two TMEM
// accumulators so the epilogue of a tile overlaps the MMAs of the next.  Warps: TMA producer, MMA issuer, 4 epilogue.
//
// X3 (the backward of the 3-pass DCN mode): each operand comes as a tf32 hi plane and a tf32 lo plane (x = hi + lo); a
// stage holds four boxes (A hi, B hi, A lo, B lo; 64 KB, so 3 stages) and each 8-wide k step issues lo.hi + hi.lo +
// hi.hi into the same accumulator: fp32-grade products, the lo.lo term (2^-22 relative) dropped.
#include "common.cuh"
#include "../../include/mrefsr_b200.h"

namespace mrefsr {

constexpr int G_BM = 128, G_BN = 128, G_BK = 32;
constexpr int G_EPI_PITCH = 36;                                    // floats per staged row (32 + 4: conflict-free 16-byte accesses)
constexpr int G_EPI_BYTES = 4 * 32 * G_EPI_PITCH * 4;              // one 32 x 32 staging tile per epilogue warp
template <bool X3> struct GemmGeom {
    static constexpr int STAGES = X3 ? 3 : 6;
    static constexpr int STAGE_BYTES = (G_BM + G_BN) * 128 * (X3 ? 2 : 1);
    static constexpr int SMEM = STAGES * STAGE_BYTES + 256 + G_EPI_BYTES + 1024;
};
static_assert(GemmGeom<true>::SMEM <= 227 * 1024, "3-pass ring exceeds shared memory");

struct GemmTcParams {
    int M, N, K;               // per batch item
    int batch;                 // batch items (per-batch mode: outputs; reduce mode: summed)
    int a_batched;             // A has a batch dimension (else the same A for every z)
    int reduce;                // 0: per-batch outputs, 1: sum over the batch, `splits` partial outputs
    int splits;
    int m_tiles, n_tiles, kblocks;   // kblocks = ceil(K / 32) per batch item
    float* D;
    long long d_stride;        // elements between outputs (per z, or per split)
    int ldd;
};

template <bool X3>
__global__ void __launch_bounds__(192, 1)
gemm_tf32_nt_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                    const __grid_constant__ CUtensorMap mapA_lo, const __grid_constant__ CUtensorMap mapB_lo,
                    const GemmTcParams prm) {
    constexpr int G_STAGES = GemmGeom<X3>::STAGES, G_STAGE_BYTES = GemmGeom<X3>::STAGE_BYTES;
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + G_STAGES * G_STAGE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + G_STAGES;
    uint64_t* tfull = bars + 2 * G_STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* epi_stage = reinterpret_cast<float*>(smem + G_STAGES * G_STAGE_BYTES + 256);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
        if (X3) {
            tma_prefetch_desc(&mapA_lo);
            tma_prefetch_desc(&mapB_lo);
        }
        for (int s = 0; s < G_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 4);
        }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<256>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int outer = prm.reduce ? prm.splits : prm.batch;
    const int total_items = outer * prm.m_tiles * prm.n_tiles;
    const long long all_kb = (long long)prm.batch * prm.kblocks;   // reduce mode: flattened (z, k-block) range
    // item -> (o, mt, nt) and its k-block range [kb0, kb1) (reduce mode: flattened over the batch)
    auto item_range = [&](int item, int& o, int& mt, int& nt, long long& kb0, long long& kb1) {
        nt = item % prm.n_tiles;
        mt = (item / prm.n_tiles) % prm.m_tiles;
        o = item / (prm.n_tiles * prm.m_tiles);
        if (prm.reduce) {
            kb0 = all_kb * o / prm.splits;
            kb1 = all_kb * (o + 1) / prm.splits;
        } else {
            kb0 = 0;
            kb1 = prm.kblocks;
        }
    };

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
                int o, mt, nt;
                long long kb0, kb1;
                item_range(item, o, mt, nt, kb0, kb1);
                for (long long kb = kb0; kb < kb1; ++kb) {
                    const int z = prm.reduce ? (int)(kb / prm.kblocks) : o;
                    const int k0 = (int)(prm.reduce ? kb % prm.kblocks : kb) * G_BK;
                    mbar_wait_backoff(&empty[stage], phase ^ 1, 32);
                    uint8_t* sa = smem + stage * G_STAGE_BYTES;
                    mbar_expect_tx(&full[stage], G_STAGE_BYTES);
                    tma_load_3d(sa, &mapA, &full[stage], k0, mt * G_BM, prm.a_batched ? z : 0);
                    tma_load_3d(sa + G_BM * 128, &mapB, &full[stage], k0, nt * G_BN, z);
                    if (X3) {
                        tma_load_3d(sa + (G_BM + G_BN) * 128, &mapA_lo, &full[stage], k0, mt * G_BM, prm.a_batched ? z : 0);
                        tma_load_3d(sa + (2 * G_BM + G_BN) * 128, &mapB_lo, &full[stage], k0, nt * G_BN, z);
                    }
                    if (++stage == G_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = umma_idesc(2, G_BM, G_BN);
            int stage = 0, it = 0;
            uint32_t phase = 0;
            for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
                int o, mt, nt;
                long long kb0, kb1;
                item_range(item, o, mt, nt, kb0, kb1);
                const int acc = it & 1;
                mbar_wait_backoff(&tempty[acc], ((it >> 1) & 1) ^ 1, 32);
                tc_fence_after();
                const uint32_t tacc = tmem_base + acc * G_BN;
                uint32_t accumulate = 0;
                for (long long kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * G_STAGE_BYTES);
                    const uint32_t sb = sa + G_BM * 128;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint64_t ah = umma_desc_sw128(sa + kk * 32, 0), bh = umma_desc_sw128(sb + kk * 32, 0);
                        if (X3) {
                            const uint32_t sal = sa + (G_BM + G_BN) * 128, sbl = sal + G_BM * 128;
                            umma_tf32(tacc, umma_desc_sw128(sal + kk * 32, 0), bh, idesc, accumulate);
                            umma_tf32(tacc, ah, umma_desc_sw128(sbl + kk * 32, 0), idesc, 1);
                            umma_tf32(tacc, ah, bh, idesc, 1);
                        } else {
                            umma_tf32(tacc, ah, bh, idesc, accumulate);
                        }
                        accumulate = 1;
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == G_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&tfull[acc]);     // (an empty k range commits at once: the epilogue then writes zeros)
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..5)
        const int q = warp & 3;                     // TMEM lane quarter this warp may access
        int it = 0;
        for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
            int o, mt, nt;
            long long kb0, kb1;
            item_range(item, o, mt, nt, kb0, kb1);
            const int acc = it & 1;
            mbar_wait_backoff(&tfull[acc], (it >> 1) & 1, 64);
            tc_fence_after();
            const int m = mt * G_BM + q * 32 + lane;
            const int n0 = nt * G_BN;
            float* drow = prm.D + (long long)o * prm.d_stride + (long long)m * prm.ldd + n0;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * G_BN;
            const bool vec = (prm.ldd & 3) == 0 && (reinterpret_cast<uintptr_t>(prm.D) & 15) == 0 && (prm.d_stride & 3) == 0;
#pragma unroll 1
            for (int c0 = 0; c0 < G_BN; c0 += 32) {
                uint32_t v[32];
                if (kb1 > kb0) {
                    tmem_ld_32x32(taddr + c0, v);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int e = 0; e < 32; ++e) v[e] = 0u;
                }
                if (vec && n0 + c0 + 32 <= prm.N) {
                    // a lane holds 32 consecutive columns of ITS row: stored directly, every 16-byte store of a warp lands in
                    // a different 128-byte line.  Through a 32 x 32 shared-memory tile instead, eight lanes cover one row's
                    // 128 bytes: full-sector, line-contiguous stores (the columns GEMM writes 6 GB per training step).
                    float* st = epi_stage + q * 32 * G_EPI_PITCH;
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        *reinterpret_cast<float4*>(st + lane * G_EPI_PITCH + e) =
                            make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]), __uint_as_float(v[e + 2]),
                                        __uint_as_float(v[e + 3]));
                    __syncwarp();
                    const int m_base = mt * G_BM + q * 32;
                    float* dbase = prm.D + (long long)o * prm.d_stride + (long long)m_base * prm.ldd + n0 + c0;
#pragma unroll
                    for (int rr = 0; rr < 8; ++rr) {
                        const int row = rr * 4 + (lane >> 3), col = (lane & 7) * 4;
                        if (m_base + row < prm.M)
                            __stcs(reinterpret_cast<float4*>(dbase + (long long)row * prm.ldd + col),
                                   *reinterpret_cast<const float4*>(st + row * G_EPI_PITCH + col));
                    }
                    __syncwarp();
                } else if (m < prm.M) {
                    {
#pragma unroll
                        for (int e = 0; e < 32; ++e)
                            if (n0 + c0 + e < prm.N) drow[c0 + e] = __uint_as_float(v[e]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<256>(tmem_base);
    }
}

// The operand pitches (lda, ldb: elements between rows) must make 16-byte multiples, the bases 16-byte aligned.
bool gemm_tc_operands_ok(const void* A, int lda, long long a_batch_stride, const void* B, int ldb, long long b_batch_stride) {
    return (reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0 && (lda & 3) == 0 &&
           (ldb & 3) == 0 && (a_batch_stride & 3) == 0 && (b_batch_stride & 3) == 0;
}

// D[o] (M x N, row pitch ldd, outputs d_stride elements apart) = A . B^T as described in the file header.
// a_batch_stride == 0: A shared by all batch items.  reduce != 0: `splits` partial outputs (see header).
// A_lo / B_lo (both or neither): the 3-pass variant, A / B are then the hi planes.
int gemm_tf32_nt(const float* A, int lda, long long a_batch_stride, const float* B, int ldb, long long b_batch_stride,
                 float* D, int ldd, long long d_stride, int M, int N, int K, int batch, int reduce, int splits,
                 cudaStream_t st, const float* A_lo, const float* B_lo) {
    MREFSR_CHECK(M > 0 && N > 0 && K > 0 && batch > 0, ERR_BAD_ARG, "gemm: bad sizes");
    MREFSR_CHECK(gemm_tc_operands_ok(A, lda, a_batch_stride, B, ldb, b_batch_stride), ERR_BAD_ARG,
                 "gemm: operands must be 16-byte aligned with row pitches that are multiples of 4 floats");
    const bool x3 = A_lo != nullptr;
    MREFSR_CHECK((B_lo != nullptr) == x3, ERR_BAD_ARG, "gemm: the 3-pass variant needs both lo planes");
    MREFSR_CHECK(!x3 || gemm_tc_operands_ok(A_lo, lda, a_batch_stride, B_lo, ldb, b_batch_stride), ERR_BAD_ARG,
                 "gemm: lo planes must be 16-byte aligned");
    const bool a_batched = a_batch_stride != 0;
    auto map_a = [&](CUtensorMap* map, const float* a) {
        return make_tensor_map_3d_strided(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a, (uint64_t)K, (uint64_t)M,
                                          a_batched ? (uint64_t)batch : 1, (uint64_t)lda * 4,
                                          (uint64_t)(a_batched ? a_batch_stride : (long long)lda * M) * 4, G_BK, G_BM,
                                          CU_TENSOR_MAP_SWIZZLE_128B);
    };
    auto map_b = [&](CUtensorMap* map, const float* b) {
        return make_tensor_map_3d_strided(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, b, (uint64_t)K, (uint64_t)N,
                                          (uint64_t)batch, (uint64_t)ldb * 4, (uint64_t)b_batch_stride * 4, G_BK, G_BN,
                                          CU_TENSOR_MAP_SWIZZLE_128B);
    };
    CUtensorMap mapA, mapB, mapA_lo, mapB_lo;
    int rc = map_a(&mapA, A);
    if (rc) return rc;
    rc = map_b(&mapB, B);
    if (rc) return rc;
    if (x3) {
        rc = map_a(&mapA_lo, A_lo);
        if (rc) return rc;
        rc = map_b(&mapB_lo, B_lo);
        if (rc) return rc;
    } else {
        mapA_lo = mapA;      // unused by the one-pass kernel
        mapB_lo = mapB;
    }
    GemmTcParams prm;
    prm.M = M;
    prm.N = N;
    prm.K = K;
    prm.batch = batch;
    prm.a_batched = a_batched ? 1 : 0;
    prm.reduce = reduce ? 1 : 0;
    prm.splits = reduce ? splits : 1;
    prm.m_tiles = cdiv(M, G_BM);
    prm.n_tiles = cdiv(N, G_BN);
    prm.kblocks = cdiv(K, G_BK);
    prm.D = D;
    prm.d_stride = d_stride;
    prm.ldd = ldd;
    const long long items = (long long)(reduce ? splits : batch) * prm.m_tiles * prm.n_tiles;
    int grid = sm_count();
    if (grid > items) grid = (int)items;
    if (x3) {
        MREFSR_CUDA(cudaFuncSetAttribute(gemm_tf32_nt_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmGeom<true>::SMEM));
        gemm_tf32_nt_kernel<true><<<grid, 192, GemmGeom<true>::SMEM, st>>>(mapA, mapB, mapA_lo, mapB_lo, prm);
    } else {
        MREFSR_CUDA(cudaFuncSetAttribute(gemm_tf32_nt_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GemmGeom<false>::SMEM));
        gemm_tf32_nt_kernel<false><<<grid, 192, GemmGeom<false>::SMEM, st>>>(mapA, mapB, mapA_lo, mapB_lo, prm);
    }
    MREFSR_LAUNCH_CHECK();
    count_launches(1);
    return 0;
}

}  // namespace mrefsr
