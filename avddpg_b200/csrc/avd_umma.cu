// avd_umma.cu -- bf16 GEMMs of the DDPG learn step on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// One CTA computes one 128 x 128 fp32 output tile: warp 0 streams 64-deep K blocks of both operands into a
// 4-stage shared-memory ring with TMA (cp.async.bulk.tensor, 128-byte swizzle), one elected thread of warp 1
// issues tcgen05.mma (M=128, N=128, K=16, bf16 x bf16 -> fp32) into a 128-column TMEM accumulator and releases
// ring slots / signals the epilogue through tcgen05.commit -> mbarrier, warps 2..5 read the accumulator back
// with tcgen05.ld (one TMEM lane = one output row per thread) and store or atomically accumulate it.
//
// Two operand layouts cover the three contractions of the learn step (SURVEY.md §8a a13):
//   TN  (forward, dgrad): A[M][K], B[N][K], both K-major        C = A B^T
//   NT  (wgrad)         : A[K][M], B[K][N], both MN-major       C += A^T B   (K = batch rows, split over CTAs)
// so activations written once as [rows][features] serve as the K-major A of the next layer's forward GEMM
// and, unchanged, as the MN-major A of the weight-gradient GEMM.
//
// Split operands (gemm_bf16x3, precision 3 of the learn step): x = hi + mid + lo with hi = bf16(x), mid = bf16(x - hi),
// lo = bf16(x - hi - mid) carries 24 significand bits, as many as fp32.  The three planes of an operand are stored
// [plane][batch][rows][inner], so plane p of batch b is batch p * batch + b of the same 3-D tensor map.  Each K block runs six
// products -- hi.hi, hi.mid, mid.hi, hi.lo, mid.mid, lo.hi; the dropped products mid.lo, lo.mid and lo.lo are below 2^-27 of
// |a||b|, under the rounding of the fp32 accumulation.  TN (PLANES = 3): one ring stage holds all six plane tiles of a K block
// (96 KB), each tile is loaded once and feeds up to three products.  NT (the weight gradient, MN-major): a K block becomes six
// virtual K blocks, one (A plane, B plane) pair each, that stream through the 4-stage ring like ordinary K blocks.  hi.hi accumulates into one TMEM tile and the five correction products into a
// second one, summed in the epilogue: the MMA's fp32 accumulation rounds once per instruction, and sharing one tile would
// round the large sum six times per K step instead of once (measured: ReLU sign flips of the learn step against fp32).
#include <utility>

#include "avd_common.cuh"
#include "avd_learn_kernels.cuh"
#include "avd_umma.cuh"

namespace avd {
namespace umma {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KB
constexpr int B_STAGE_BYTES = BN * BK * 2;   // 16 KB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int SCRATCH_BYTES = 4 * 32 * 33 * 4;   // per-epilogue-warp transpose scratch
// planes = 3 (six-tile stages): the epilogue's transpose scratch reuses the ring, which is idle once the accumulator is complete
constexpr int smem_bytes(int stages, int bn = BN, int planes = 1) {
    return stages * planes * (A_STAGE_BYTES + bn * BK * 2) + 1024 /*align slack*/ + 256 /*barriers*/ + (planes == 1 ? SCRATCH_BYTES : 0);
}
// TN GEMMs of the learn step have K <= 320 (2..5 k-blocks): 2 stages = 82 KB so that two CTAs share an SM and one
// CTA's prologue/epilogue overlaps another's MMAs; the NT weight-gradient GEMM streams thousands of rows: 4 stages (one CTA
// per SM).  Split-operand TN: ONE six-tile stage (97 KB) so that two CTAs (2 x 256 TMEM columns) share an SM and overlap --
// measured at the C2 learn shape, two six-tile stages and one CTA per SM ran the TN GEMMs 6 % slower than six pair-stages.
constexpr int STAGES_TN = 2, STAGES_NT = 4, STAGES_TN3 = 1;
constexpr int NUM_THREADS = 192;             // warp 0 TMA, warp 1 MMA (+TMEM alloc), warps 2..5 epilogue

struct GemmParams {
    int M, N;              // valid output rows / columns (per batch)
    int k_blocks;          // number of 64-deep K blocks per split
    int splitk;
    float* C;
    int64_t ldc, c_batch;
    int atomic;            // 1: atomicAdd into C (split-K)
    int n_fastest;         // 1: blockIdx.x walks the N tiles, so the CTAs that share an A tile run together and re-read it from L2
    uint32_t a_fmt, b_fmt; // operand formats of the kind::f16 MMA: FMT_F16 / FMT_BF16, chosen independently
    int pairs;             // 1: plain operands; 6: split operands, six (A plane, B plane) products per K block
    int batch;             // batches per plane: plane p of batch b is tensor-map batch p * batch + b
};

// plane of A / B in product 0..5 of a split K block (2 bits each): hi.hi, hi.mid, mid.hi, hi.lo, mid.mid, lo.hi
constexpr uint32_t kPairA = (1u << 4) | (1u << 8) | (2u << 10), kPairB = (1u << 2) | (2u << 6) | (1u << 8);

// PLANES = 3: split operands (g.pairs = 6), every stage holds the three planes of A and of B for one K block
template <bool MN_MAJOR, int STAGES, int BN_, int PLANES = 1>
__global__ void __launch_bounds__(NUM_THREADS, PLANES == 3 ? 2 : (STAGES <= 2) ? 3 : 1) gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                   const __grid_constant__ CUtensorMap tmB, GemmParams g) {
    constexpr int B_STAGE = BN_ * BK * 2;
    constexpr int STAGE = PLANES * (A_STAGE_BYTES + B_STAGE);
    constexpr int PPS = PLANES == 3 ? 6 : 1;      // products per stage
    static_assert(BN_ == 128 || (BN_ == 64 && MN_MAJOR), "64-wide output tiles exist for the MN-major layout only");
    static_assert(PLANES == 1 || (PLANES == 3 && !MN_MAJOR), "six-tile stages exist for the TN layout only");
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);   // SWIZZLE_128B tiles need 1024-byte alignment
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* accum_bar = empty_bar + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
    float* scratch_all = reinterpret_cast<float*>(PLANES == 3 ? smem : smem + STAGES * STAGE + 256);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = (g.n_fastest ? blockIdx.y : blockIdx.x) * BM, n0 = (g.n_fastest ? blockIdx.x : blockIdx.y) * BN_;
    const int batch = blockIdx.z / g.splitk, split = blockIdx.z % g.splitk;
    const int kb0 = split * g.k_blocks;
    const int nv = PLANES == 3 ? g.k_blocks : g.k_blocks * g.pairs;   // ring stages this CTA streams

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(accum_bar, 1);
        fence_barrier_init();
    }
    const uint32_t tmem_cols = g.pairs > 1 ? 2 * BN : BN;   // split operands: hi.hi tile at column 0, corrections at column BN
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            for (int v = 0; v < nv; ++v) {     // PLANES = 1: virtual K block v = K block v / pairs, product v % pairs
                const int s = v % STAGES;
                const uint32_t ph = (v / STAGES) & 1;
                const int kb = PLANES == 3 ? v : v / g.pairs, pr = PLANES == 3 ? 0 : v - kb * g.pairs;
                const int za = batch + g.batch * (int)((kPairA >> (2 * pr)) & 3u), zb = batch + g.batch * (int)((kPairB >> (2 * pr)) & 3u);
                mbar_wait(&empty_bar[s], ph ^ 1);
                uint8_t* sa = smem + s * STAGE;
                uint8_t* sb = sa + PLANES * A_STAGE_BYTES;
                mbar_expect_tx(&full_bar[s], STAGE);
                const int k = (kb0 + kb) * BK;
                if (PLANES == 3) { // planes hi, mid, lo of A, then of B
#pragma unroll
                    for (int pl = 0; pl < 3; ++pl) {
                        tma_load_3d(sa + pl * A_STAGE_BYTES, &tmA, &full_bar[s], k, m0, batch + g.batch * pl);
                        tma_load_3d(sb + pl * B_STAGE, &tmB, &full_bar[s], k, n0, batch + g.batch * pl);
                    }
                } else if (!MN_MAJOR) {   // box {64 k, 128 rows}
                    tma_load_3d(sa, &tmA, &full_bar[s], k, m0, za);
                    tma_load_3d(sb, &tmB, &full_bar[s], k, n0, zb);
                } else {           // box {64 mn, 64 k-rows}; two MN chunks per operand
                    tma_load_3d(sa, &tmA, &full_bar[s], m0, k, za);
                    tma_load_3d(sa + A_STAGE_BYTES / 2, &tmA, &full_bar[s], m0 + 64, k, za);
                    tma_load_3d(sb, &tmB, &full_bar[s], n0, k, zb);
                    if (BN_ == 128) tma_load_3d(sb + B_STAGE / 2, &tmB, &full_bar[s], n0 + 64, k, zb);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            const uint32_t idesc = make_idesc_f16kind(BM, BN_, MN_MAJOR, MN_MAJOR, g.a_fmt, g.b_fmt);
            for (int v = 0; v < nv; ++v) {
                const int s = v % STAGES;
                const uint32_t ph = (v / STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                const uint32_t s0 = smem_u32(smem + s * STAGE);
#pragma unroll
                for (int q = 0; q < PPS; ++q) {
                    const int kb = PLANES == 3 ? v : v / g.pairs, pr = PLANES == 3 ? q : v - kb * g.pairs;
                    const uint32_t dtile = tmem_base + (pr ? (uint32_t)BN : 0u);
                    const bool first = kb == 0 && pr <= 1;     // first K step into this tile overwrites it
                    // PLANES = 3: this product's A / B plane tiles inside the stage; PLANES = 1: the stage holds one pair
                    const uint32_t sa = s0 + (PLANES == 3 ? ((kPairA >> (2 * pr)) & 3u) * A_STAGE_BYTES : 0u);
                    const uint32_t sb = s0 + PLANES * A_STAGE_BYTES + (PLANES == 3 ? ((kPairB >> (2 * pr)) & 3u) * B_STAGE : 0u);
#pragma unroll
                    for (int j = 0; j < BK / 16; ++j) {
                        uint64_t ad, bd;
                        if (!MN_MAJOR) {   // advance 16 bf16 = 32 B along K inside the 128-byte swizzle row
                            ad = make_smem_desc(sa + j * 32, 16, 1024);
                            bd = make_smem_desc(sb + j * 32, 16, 1024);
                        } else {           // advance 16 K rows = two 8-row groups of 1024 B; MN chunks 8 KB apart
                            ad = make_smem_desc(sa + j * 2048, A_STAGE_BYTES / 2, 1024);
                            bd = make_smem_desc(sb + j * 2048, BN_ == 128 ? B_STAGE / 2 : 16, 1024);
                        }
                        mma_bf16(dtile, ad, bd, idesc, !first || j != 0);
                    }
                }
                mma_commit(&empty_bar[s]);     // slot free once these MMAs have read it
            }
            mma_commit(accum_bar);             // accumulator complete
        }
    } else {  // ===== epilogue: warps 2..5, TMEM lane quadrant = warp % 4 =====
        const int q = warp & 3;
        mbar_wait(accum_bar, 0);
        tc_fence_after();
        const int row = m0 + q * 32 + lane;
        float* crow = g.C + (int64_t)batch * g.c_batch + (int64_t)row * g.ldc;
        float* scratch = scratch_all + (warp - 2) * (32 * 33);
        float* cblock = g.C + (int64_t)batch * g.c_batch + (int64_t)(m0 + q * 32) * g.ldc;
        const int rows_here = min(32, g.M - (m0 + q * 32));
#pragma unroll 1
        for (int c = 0; c < BN_ / 32; ++c) {
            const int col0 = n0 + c * 32;
            if (col0 >= g.N) break;
            float v[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
            if (g.pairs > 1) {
                float w[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(BN + c * 32), w);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += w[j];
            }
            if (g.atomic) {
                if (row < g.M) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (col0 + j < g.N) atomicAdd(crow + col0 + j, v[j]);
                }
            } else if (rows_here > 0) {
                store_block_32x32(scratch, v, cblock + col0, g.ldc, rows_here, min(32, g.N - col0), lane);
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// planes = 1: plain 16-bit operands; planes = 3: bf16 hi / mid / lo planes, plane p of batch b at A + (p * batch + b) * a_batch
static int launch_gemm(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B, int64_t ldb,
                       int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, int a_fmt, int b_fmt, int planes, cudaStream_t st) {
    AVD_REQUIRE(layout == 0 || layout == 1, "layout must be 0 (TN) or 1 (NT)");
    AVD_REQUIRE(batch >= 1 && M >= 1 && N >= 1 && K >= 1 && splitk >= 1, "bad GEMM sizes");
    AVD_REQUIRE(A && B && C, "null operand");
    AVD_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && a_batch % 8 == 0 && b_batch % 8 == 0, "bf16 leading dimensions must be multiples of 8 elements (16 B)");
    AVD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0, "operands must be 16-byte aligned");
    static bool attr_set = false;
    if (!attr_set) {
        AVD_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<false, STAGES_TN, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(STAGES_TN)));
        AVD_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<false, STAGES_TN3, 128, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         smem_bytes(STAGES_TN3, BN, 3)));
        AVD_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<true, STAGES_NT, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(STAGES_NT)));
        AVD_CUDA_OK(cudaFuncSetAttribute(gemm_bf16_kernel<true, STAGES_NT, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(STAGES_NT, 64)));
        attr_set = true;
    }
    CUtensorMap tmA, tmB;
    const int kblocks_total = (K + BK - 1) / BK;
    if (splitk > kblocks_total) splitk = kblocks_total;
    GemmParams g;
    g.M = M; g.N = N; g.splitk = splitk;
    g.k_blocks = (kblocks_total + splitk - 1) / splitk;
    g.C = C; g.ldc = ldc; g.c_batch = c_batch; g.atomic = (splitk > 1 || layout == 1) ? 1 : 0;
    g.a_fmt = (uint32_t)a_fmt; g.b_fmt = (uint32_t)b_fmt;
    g.pairs = planes == 3 ? 6 : 1;
    g.batch = batch;
    const bool narrow = layout == 1 && N <= 64;     // narrow outputs: one 64-column MN chunk of B per stage
    const int bn = narrow ? 64 : BN;
    dim3 grid((M + BM - 1) / BM, (N + bn - 1) / bn, batch * splitk);
    g.n_fastest = (layout == 0 && grid.y > 1 && grid.x <= 65535) ? 1 : 0;
    if (g.n_fastest) std::swap(grid.x, grid.y);
    const int zmaps = planes * batch;
    if (layout == 0) {
        if (int rc = make_tensor_map(&tmA, A, K, M, zmaps, lda, a_batch, BK, BM)) return rc;
        if (int rc = make_tensor_map(&tmB, B, K, N, zmaps, ldb, b_batch, BK, BN)) return rc;
        if (planes == 3) gemm_bf16_kernel<false, STAGES_TN3, 128, 3><<<grid, NUM_THREADS, smem_bytes(STAGES_TN3, BN, 3), st>>>(tmA, tmB, g);
        else gemm_bf16_kernel<false, STAGES_TN, 128><<<grid, NUM_THREADS, smem_bytes(STAGES_TN), st>>>(tmA, tmB, g);
    } else {
        if (int rc = make_tensor_map(&tmA, A, M, K, zmaps, lda, a_batch, 64, BK)) return rc;
        if (int rc = make_tensor_map(&tmB, B, N, K, zmaps, ldb, b_batch, 64, BK)) return rc;
        if (narrow) gemm_bf16_kernel<true, STAGES_NT, 64><<<grid, NUM_THREADS, smem_bytes(STAGES_NT, 64), st>>>(tmA, tmB, g);
        else gemm_bf16_kernel<true, STAGES_NT, 128><<<grid, NUM_THREADS, smem_bytes(STAGES_NT), st>>>(tmA, tmB, g);
    }
    AVD_LAUNCH_OK();
    return AVD_OK;
}

int gemm_f16kind(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B, int64_t ldb,
                 int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, int a_fmt, int b_fmt, cudaStream_t st) {
    AVD_REQUIRE((a_fmt == 0 || a_fmt == 1) && (b_fmt == 0 || b_fmt == 1), "operand formats: 0 = fp16, 1 = bf16");
    if (a_fmt != b_fmt) {       // the instruction descriptor can express it, the B200 tensor pipe traps on it (illegal instruction)
        set_error("kind::f16 MMAs need both operands in the same 16-bit format (got A %s, B %s)", a_fmt ? "bf16" : "fp16", b_fmt ? "bf16" : "fp16");
        return AVD_ERR_UNSUPPORTED;
    }
    return launch_gemm(layout, batch, M, N, K, A, lda, a_batch, B, ldb, b_batch, C, ldc, c_batch, splitk, a_fmt, b_fmt, 1, st);
}

int gemm_bf16(int planes, int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B, int64_t ldb,
              int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, cudaStream_t st) {
    AVD_REQUIRE(planes == 1 || (a_batch > 0 && b_batch > 0),
                "split operands need positive batch strides (plane p of batch b starts at (p * batch + b) * stride)");
    return launch_gemm(layout, batch, M, N, K, A, lda, a_batch, B, ldb, b_batch, C, ldc, c_batch, splitk, (int)FMT_BF16, (int)FMT_BF16, planes, st);
}

}  // namespace umma
}  // namespace avd

extern "C" int avd_gemm_f16kind(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B,
                                int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, int a_fmt, int b_fmt,
                                void* stream) {
    return avd::umma::gemm_f16kind(layout, batch, M, N, K, A, lda, a_batch, B, ldb, b_batch, C, ldc, c_batch, splitk, a_fmt, b_fmt,
                                   (cudaStream_t)stream);
}

extern "C" int avd_gemm_bf16(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B,
                             int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, void* stream) {
    return avd::umma::gemm_bf16(1, layout, batch, M, N, K, A, lda, a_batch, B, ldb, b_batch, C, ldc, c_batch, splitk, (cudaStream_t)stream);
}

extern "C" int avd_gemm_bf16x3(int layout, int batch, int M, int N, int K, const void* A_planes, int64_t lda, int64_t a_batch, const void* B_planes,
                               int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, void* stream) {
    return avd::umma::gemm_bf16(3, layout, batch, M, N, K, A_planes, lda, a_batch, B_planes, ldb, b_batch, C, ldc, c_batch, splitk,
                                (cudaStream_t)stream);
}
