// avd_dgrad3.cu -- layer-1 backward of the DDPG learn step as ONE persistent tensor-core kernel (sm_100a):
//
//   dz2 tile [128 rows][128] (bf16, TMA)  --tcgen05.mma against W2' (resident in shared memory, 64-feature chunks)-->
//   dR chunk [128 rows][64 features] in TMEM  --epilogue warps: ReLU sign mask, bf16-->  dz1 chunk in shared memory
//   --tcgen05.mma  dz1^T [x_hi | 1 | x_lo]  (MN-major A = the chunk just written, K = the 128 rows)-->  G1 accumulators
//   that stay in TMEM for the whole kernel and are added to global memory once per CTA.
//
// dz1 never reaches HBM: per row the kernel reads 256 B (dz2) + 40 B (masks) + 32 B (x) and writes nothing.
//   G1[f][c] = sum_n dz1[n][f] xext[n][c]  =>  dW1[k][f] = G1[f][k] + G1[f][8+k],  dWa[f] = G1[l1+f][4] + G1[l1+f][12],
//   db1[f] = G1[f][5]                                                    (unfold_kernel in avd_ddpg.cu)
// Math: dR = dz2 W2'^T with W2' = diag(sc1) W2 (BatchNorm folded, pack_fold_kernel), dz1 = dR [z1 > 0]
// (workers/trainer.py:498, 506 through agent/model.py:19-33, 62-77).
//
// Warps: 0 issuer of the dR chunk MMAs, 18 issuer of the G1 / db2 MMAs, 1 TMA producer, 2..17 epilogue (TMEM lane quadrant = warp % 4, 32 of a chunk pair's 128 columns each).  TMEM: 3-slot ring of 128-column dR chunk pairs + 3 x 16 columns of G1 + 16 columns of
// dz2^T xext, whose column 5 (xext's constant one) is the layer-2 bias gradient db2.
#include "avd_common.cuh"
#include "avd_learn_kernels.cuh"
#include "avd_umma.cuh"

namespace avd {
namespace dgrad3 {

using namespace umma;

constexpr int TILE_M = 128, L2N = 128, KB = 64, MAX_NC = 5, NRING = 3;
constexpr int NUM_THREADS = 32 * 19;
constexpr int WARP_G1 = 18;                                  // issuer of the G1 / db2 MMAs
constexpr int WCHUNK_BYTES = 64 * 128;                       // one 64-feature x 64-k block of W2': 8 KB
constexpr int OFF_W = 0;                                     // [2 k-blocks][5 chunks][64 rows][128 B] = 80 KB
constexpr int OFF_A = OFF_W + 2 * MAX_NC * WCHUNK_BYTES;     // 2 dz2 tiles of 32 KB (released as soon as the chunk MMAs have read them)
constexpr int A_BYTES = 2 * TILE_M * 128;
constexpr int OFF_XT = OFF_A + 2 * A_BYTES;                  // 4 xext^T tiles of 4 KB (read last, by the G1 MMAs): deeper ring
constexpr int XT_BYTES = 2 * 16 * 128, NXT = 4;
constexpr int OFF_ST = OFF_XT + NXT * XT_BYTES;              // 2 pair buffers x 2 chunks x 16 KB
constexpr int OFF_BAR = OFF_ST + 4 * TILE_M * 128;
constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");
static_assert(A_BYTES % 1024 == 0 && XT_BYTES % 1024 == 0 && OFF_ST % 1024 == 0, "swizzled tiles need 1024-byte alignment");

struct Args {
    int A, F, NC;               // agents, layer-1 features (256 or 256 + la), 64-column chunks
    int64_t R;
    const uint32_t* mask;       // [A*R][mask_words]
    int mask_words;
    float* G1;                  // partial slice of CTA (agent, cta): G1 + (agent*ctas_per_agent + cta)*Fp*16, [Fp][16]
    int Fp;
    float* db2;                 // [A][db2_stride] += sum_n dz2[n][j]   (layer-2 bias gradient)
    int64_t db2_stride;
    int tiles_per_agent, ctas_per_agent;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// NC: 64-feature chunks of layer 1: 4 (actor, 256 features) or 5 (critic, 256 + action features).  F16 (precision = 2): every
// operand -- dz2 tile, W2'', the staged dz1 chunks and the hi/lo-split x_ext -- is fp16 instead of bf16 (no mixed-format MMA on B200).
template <int NC, bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1) dgrad3_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmDZ,
                                                                const __grid_constant__ CUtensorMap tmXT, Args g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* d_full = reinterpret_cast<uint64_t*>(smem + OFF_BAR);   // [3]
    uint64_t* d_empty = d_full + NRING;                               // [3]
    uint64_t* st_full = d_empty + NRING;                              // [2]
    uint64_t* st_empty = st_full + 2;                                 // [2]
    uint64_t* a_full = st_empty + 2;                                  // [2]
    uint64_t* a_empty = a_full + 2;                                   // [2]
    uint64_t* xt_full = a_empty + 2;                                  // [4]
    uint64_t* xt_empty = xt_full + NXT;                               // [4]
    uint64_t* w_full = xt_empty + NXT;
    uint64_t* g1_done = w_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(g1_done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int agent = (int)blockIdx.x / g.ctas_per_agent;
    const int cta = (int)blockIdx.x - agent * g.ctas_per_agent;
    const int T = (g.tiles_per_agent - cta + g.ctas_per_agent - 1) / g.ctas_per_agent;
    constexpr int NP = (NC + 1) >> 1;                  // chunk pairs (the last pair of the critic has one chunk)

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmW); tma_prefetch_desc(&tmDZ); tma_prefetch_desc(&tmXT);
        for (int i = 0; i < NRING; ++i) { mbar_init(&d_full[i], 1); mbar_init(&d_empty[i], 16); }
        for (int i = 0; i < 2; ++i) { mbar_init(&st_full[i], 16); mbar_init(&st_empty[i], 1); mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 2); }
        for (int i = 0; i < NXT; ++i) { mbar_init(&xt_full[i], 1); mbar_init(&xt_empty[i], 1); }
        mbar_init(w_full, 1);
        mbar_init(g1_done, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                      // dz2, the sign masks and the partial-slice buffers belong to earlier launches until here
    pdl_launch_dependents();
    auto tile_of = [&](int tc) { return cta + tc * g.ctas_per_agent; };
    // Chunk pair p of local tile t has the running index pk = t NP + p: TMEM ring slot pk % 3 (128 columns), staging buffer pk & 1.

    if (warp == 0 || warp == WARP_G1) {
        // ================================================ MMA issuers ================================================
        // Warp-uniform control flow, tcgen05 instructions predicated on one elected lane (see avd_umma.cuh).  A tcgen05.mma
        // issues at the pace of the tensor pipe and every tcgen05.commit costs its thread ~140 cycles; one thread issuing all
        // 56 MMAs and 6 commits of a tile was busy ~80 % of the kernel, so the two products have an issuer warp each:
        //   warp 0:  dR chunk pairs (N = 128)             warp 18:  db2 and G1 (N = 16), which read what the epilogue staged.
        // A tcgen05.commit only tracks the MMAs of its own thread, so the dz2 tile is handed back by both (a_empty counts 2).
        if (T > 0) {
            const uint32_t leader = elect_one();
            constexpr uint32_t FOP = F16 ? FMT_F16 : FMT_BF16;
            constexpr uint32_t idesc_2 = make_idesc_f16kind(TILE_M, 128, false, false, FOP, FOP);   // dz2 (K-major) x W2'' chunk pair (K-major)
            constexpr uint32_t idesc_1 = make_idesc_f16kind(TILE_M, 64, false, false, FOP, FOP);    // ... x single chunk
            constexpr uint32_t idesc_g = make_idesc_f16kind(TILE_M, 16, true, false, FOP, FOP);     // dz1 / dz2 (MN-major) x xext^T (K-major)
            const uint64_t dA = make_smem_desc(smem_u32(smem + OFF_A), 16, 1024);                 // dz2 tile as K-major A
            const uint64_t dAt = make_smem_desc(smem_u32(smem + OFF_A), TILE_M * 128, 1024);      // dz2 tile as MN-major A (two 64-column halves)
            const uint64_t dW = make_smem_desc(smem_u32(smem + OFF_W), 16, 1024);
            const uint64_t dX = make_smem_desc(smem_u32(smem + OFF_XT), 16, 1024);
            const uint64_t dS = make_smem_desc(smem_u32(smem + OFF_ST), TILE_M * 128, 1024);      // staged dz1 chunk pair as MN-major A
            if (warp == 0) {
                // dR of chunk pair p of local tile t = dz2 tile . W2'[128 p .. 128 p + 127]^T  -> ring slot pk % 3
                mbar_wait(w_full, 0);
                uint32_t rs = 0, rph = 0;
                for (int t = 0; t < T; ++t) {
                    const uint32_t a_off = (uint32_t)(t & 1) * A_BYTES;
                    mbar_wait(&a_full[t & 1], ((uint32_t)t >> 1) & 1);
#pragma unroll
                    for (int p = 0; p < NP; ++p) {
                        const bool both = 2 * p + 1 < NC;
                        mbar_wait(&d_empty[rs], rph ^ 1);
                        tc_fence_after();
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks)
                            mma_bf16_p(leader, tmem_base + rs * 128, desc_add(dA, a_off + (ks >> 2) * (TILE_M * 128) + (ks & 3) * 32),
                                       desc_add(dW, (uint32_t)((ks >> 2) * MAX_NC + 2 * p) * WCHUNK_BYTES + (ks & 3) * 32), both ? idesc_2 : idesc_1, ks != 0);
                        mma_commit_p(leader, &d_full[rs]);
                        if (++rs == NRING) { rs = 0; rph ^= 1; }
                    }
                    mma_commit_p(leader, &a_empty[t & 1]);      // all chunk MMAs of this tile have read the dz2 tile
                }
            } else {
                uint32_t pk = 0;
                for (int t = 0; t < T; ++t) {
                    const uint32_t a_off = (uint32_t)(t & 1) * A_BYTES, x_off = (uint32_t)(t % NXT) * XT_BYTES;
                    mbar_wait(&a_full[t & 1], ((uint32_t)t >> 1) & 1);
                    mbar_wait(&xt_full[t % NXT], ((uint32_t)t / NXT) & 1);
                    tc_fence_after();
                    // db2[j] = sum_n dz2[n][j]: the dz2 tile read as an MN-major A operand against the constant-one column (5) of xext
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        mma_bf16_p(leader, tmem_base + 432u, desc_add(dAt, a_off + ks * 2048), desc_add(dX, x_off + (ks >> 2) * (16 * 128) + (ks & 3) * 32),
                                   idesc_g, (t | ks) != 0);
                    mma_commit_p(leader, &a_empty[t & 1]);
                    // G1[128 p ..] += (staged dz1 chunk pair)^T . xext tile
#pragma unroll
                    for (int p = 0; p < NP; ++p) {
                        const uint32_t sb = pk & 1;
                        mbar_wait(&st_full[sb], (pk >> 1) & 1);
                        tc_fence_after();
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks)
                            mma_bf16_p(leader, tmem_base + 384u + (uint32_t)(p * 16), desc_add(dS, sb * (2 * TILE_M * 128) + ks * 2048),
                                       desc_add(dX, x_off + (ks >> 2) * (16 * 128) + (ks & 3) * 32), idesc_g, (t | ks) != 0);
                        mma_commit_p(leader, &st_empty[sb]);
                        ++pk;
                    }
                    mma_commit_p(leader, &xt_empty[t % NXT]);   // db2 and G1 of this tile have read the x_ext tile
                }
                mma_commit_p(leader, g1_done);
            }
        }
    } else if (warp == 1) {
        // ================================================ TMA producer ================================================
        if (T > 0) {
            const uint32_t leader = elect_one();
            mbar_expect_tx_p(leader, w_full, (uint32_t)(2 * NC * WCHUNK_BYTES));
            for (int kb = 0; kb < 2; ++kb)
                for (int c = 0; c < NC; ++c) tma_load_3d_p(leader, smem + OFF_W + (kb * MAX_NC + c) * WCHUNK_BYTES, &tmW, w_full, kb * KB, c * 64, agent);
            for (int t = 0; t < T; ++t) {
                const int b = t & 1, xb = t % NXT;
                const int r0 = tile_of(t) * TILE_M;
                mbar_wait(&xt_empty[xb], (((uint32_t)t / NXT) & 1) ^ 1);
                uint8_t* xdst = smem + OFF_XT + xb * XT_BYTES;
                mbar_expect_tx_p(leader, &xt_full[xb], XT_BYTES);
                tma_load_3d_p(leader, xdst, &tmXT, &xt_full[xb], r0, 0, agent);
                tma_load_3d_p(leader, xdst + 16 * 128, &tmXT, &xt_full[xb], r0 + KB, 0, agent);
                mbar_wait(&a_empty[b], (((uint32_t)t >> 1) & 1) ^ 1);
                uint8_t* dst = smem + OFF_A + b * A_BYTES;
                mbar_expect_tx_p(leader, &a_full[b], A_BYTES);
                tma_load_3d_p(leader, dst, &tmDZ, &a_full[b], 0, r0, agent);
                tma_load_3d_p(leader, dst + TILE_M * 128, &tmDZ, &a_full[b], KB, r0, agent);
            }
        }
    } else {
        // ================================================== epilogue ==================================================
        // All 16 warps work on the SAME chunk pair: TMEM lane quadrant q, 32-column quarter c4 of the pair's 128 columns.  One
        // warp alone issues a dependent instruction only every few cycles, so short per-thread streams (32 columns) and many
        // warps per pair matter more than keeping several pairs in flight.
        const int q = warp & 3, c4 = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = (uint32_t)(q * 32) << 16;
        // The sign mask word of the next pair is fetched while the current pair is processed (a load issued right before its use
        // would put a full global-memory latency on every pair), from a per-tile row pointer: the epilogue warps are bound by
        // instruction issue, so the per-pair bookkeeping is kept to a handful of instructions.
        auto mask_row = [&](int t) -> const uint32_t* {
            const int64_t r_in = (int64_t)tile_of(t) * TILE_M + row;
            const int64_t nrow = (int64_t)agent * g.R + (r_in < g.R ? r_in : g.R - 1);
            return g.mask + nrow * g.mask_words + c4;           // word 4 p + c4 of the row = columns 128 p + 32 c4 ..
        };
        const uint32_t* mrow = T > 0 ? mask_row(0) : g.mask;
        uint32_t neg_next = T > 0 ? __ldg(mrow) : 0u;
        uint32_t rs = 0, rph = 0, pk = 0;                        // TMEM ring slot and its phase, running pair index
        for (int t = 0; t < T; ++t) {
            const uint32_t* mrow_next = t + 1 < T ? mask_row(t + 1) : mrow;
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                const uint32_t sb = pk & 1;
                const bool work = 2 * p + (c4 >> 1) < NC;        // the second chunk of a lone last pair does not exist
                const uint32_t neg = neg_next;
                if (p + 1 < NP) neg_next = (2 * (p + 1) + (c4 >> 1) < NC) ? __ldg(mrow + 4 * (p + 1)) : 0u;
                else neg_next = __ldg(mrow_next);
                mbar_wait(&d_full[rs], rph);
                tc_fence_after();
                uint32_t pkd[16];            // the masked quarter as bf16 pairs: the TMEM slot is released before the staging buffer is needed
                if (work) {
                    float v[32];
                    tmem_ld32(tmem_base + rs * 128 + (uint32_t)(c4 * 32) + tlane, v);
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (neg & (0x80000000u >> j)) v[j] = 0.0f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) pkd[j] = pack_x2<F16>(v[2 * j], v[2 * j + 1]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&d_empty[rs]);
                mbar_wait(&st_empty[sb], ((pk >> 1) & 1) ^ 1);
                if (work) {
                    uint8_t* srow = smem + OFF_ST + sb * (2 * TILE_M * 128) + (c4 >> 1) * (TILE_M * 128) + row * 128;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        *reinterpret_cast<uint4*>(srow + ((((c4 & 1) * 4 + kk) ^ (row & 7)) << 4)) =
                            make_uint4(pkd[4 * kk], pkd[4 * kk + 1], pkd[4 * kk + 2], pkd[4 * kk + 3]);
                    fence_proxy_async();
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&st_full[sb]);
                ++pk;
                if (++rs == NRING) { rs = 0; rph ^= 1; }
            }
            mrow = mrow_next;
        }
        const int grp = c4;
        // ---- G1 accumulators of this CTA -> global (features p*128 + row, 16 columns)
        if (grp == 0 && T > 0) {
            mbar_wait(g1_done, 0);
            tc_fence_after();
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                float v[16];
                tmem_ld16(tmem_base + 384u + (uint32_t)(p * 16) + tlane, v);
                const int f = p * 128 + row;
                if (f < g.F) {           // plain stores into this CTA's slice (summed by the unfold kernel)
                    float* dst = g.G1 + (((int64_t)agent * g.ctas_per_agent + cta) * g.Fp + f) * 16;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
            tc_fence_before();
        }
        if (grp == 1 && T > 0) {             // layer-2 bias gradient: column 5 of the dz2^T xext accumulator, lane = j
            mbar_wait(g1_done, 0);
            tc_fence_after();
            float v[16];
            tmem_ld16(tmem_base + 432u + tlane, v);
            atomicAdd(g.db2 + (int64_t)agent * g.db2_stride + row, v[5]);
            tc_fence_before();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// DZ: 16-bit [A*R][128];  W2b: [A][F][128] folded layer-2 kernel W2'' = W2' diag(w3') (bf16, or with f16 = true everything fp16, W2b
// scaled by a power of two s per agent and DZ by dm_scale: G1 / db2 then carry those factors, which the unfold kernel divides out);  mask: [A*R][mask_words];  xextT: bf16 [A][16][Rp]
// (Rp = rows per agent rounded up to a multiple of 64);  G1: fp32 [A][ctas_per_agent][Fp][16] partial slices, one per CTA, plain
// stores (rows < F; the caller sums them);  db2: fp32 [A][db2_stride] (first 128 entries), accumulated into (zero it first).
int run(bool f16, int A, int64_t R, int F, const bf16* DZ, const bf16* W2b, const uint32_t* mask, int mask_words, const bf16* xextT, int64_t Rp, float* G1,
        int Fp, float* db2, int64_t db2_stride, cudaStream_t st) {
    AVD_REQUIRE(A >= 1 && R >= 1 && F > 192 && F % 16 == 0 && F <= MAX_NC * 64 && Fp >= F, "bad sizes for the fused dgrad kernel");
    AVD_REQUIRE(DZ && W2b && mask && xextT && G1 && db2 && Rp % 64 == 0 && Rp >= R, "null buffer / bad pitch");
    static bool attr_set = false;
    if (!attr_set) {
        AVD_CUDA_OK(cudaFuncSetAttribute(dgrad3_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        AVD_CUDA_OK(cudaFuncSetAttribute(dgrad3_kernel<5, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        AVD_CUDA_OK(cudaFuncSetAttribute(dgrad3_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        AVD_CUDA_OK(cudaFuncSetAttribute(dgrad3_kernel<5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    CUtensorMap tmW, tmDZ, tmXT;
    if (int rc = make_tensor_map(&tmW, W2b, L2N, (uint64_t)F, (uint64_t)A, L2N, (uint64_t)F * L2N, KB, 64)) return rc;
    if (int rc = make_tensor_map(&tmDZ, DZ, L2N, (uint64_t)R, (uint64_t)A, L2N, (uint64_t)R * L2N, KB, TILE_M)) return rc;
    if (int rc = make_tensor_map(&tmXT, xextT, (uint64_t)R, 16, (uint64_t)A, (uint64_t)Rp, (uint64_t)16 * Rp, KB, 16)) return rc;
    Args g;
    g.A = A; g.F = F; g.NC = (F + 63) / 64; g.R = R; g.mask = mask; g.mask_words = mask_words; g.G1 = G1; g.Fp = Fp; g.db2 = db2; g.db2_stride = db2_stride;
    g.tiles_per_agent = (int)((R + TILE_M - 1) / TILE_M);
    g.ctas_per_agent = ctas_per_agent(A, R);
    const unsigned grid = (unsigned)(g.ctas_per_agent * A);
    if (g.NC == 4 && !f16) AVD_CUDA_OK(launch_pdl(dgrad3_kernel<4, false>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tmW, tmDZ, tmXT, g));
    else if (!f16) AVD_CUDA_OK(launch_pdl(dgrad3_kernel<5, false>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tmW, tmDZ, tmXT, g));
    else if (g.NC == 4) AVD_CUDA_OK(launch_pdl(dgrad3_kernel<4, true>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tmW, tmDZ, tmXT, g));
    else AVD_CUDA_OK(launch_pdl(dgrad3_kernel<5, true>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tmW, tmDZ, tmXT, g));
    AVD_LAUNCH_OK();
    return AVD_OK;
}

}  // namespace dgrad3
}  // namespace avd
