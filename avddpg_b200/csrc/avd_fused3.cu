// avd_fused3.cu -- one persistent kernel per network pass of the DDPG learn step (sm_100a): layer 1, layer 2, head and --
// for the passes that are differentiated -- the head backward, all on one 128-row tile at a time without HBM round trips.
//
//   x (4 state words [+ action])  --tcgen05.mma, hi/lo-split bf16, K = 16-->  z1 (TMEM)
//   --consumer warps-->  r1 = relu(z1) as bf16 into the 128B-swizzled K-major A tile (+ sign bits for the ReLU backward)
//   --tcgen05.mma against the BN-folded W2'^T (resident in shared memory)-->  z2 (TMEM, double buffered)
//   --pass 1-->  q = relu(z2 + b2') . w3' + b3'       (row sum split over four warps, combined through shared memory)
//   --pass 2 (backward modes)-->  dq from the loss, dm = dq [z2 + b2' > 0] as bf16 into a shared-memory tile (dz2 = dm diag(w3'):
//        the head weight is folded into the dgrad operand and into the unfold of the weight gradient, which also yields
//        U[j] = sum_n dq_n relu(z2)[n][j] for the head / BN2 weight gradients),  per-thread partial sums of  sum dq  and the loss
//   --TMA store-->  the dm tile to HBM for the weight-gradient kernel (avd_wgrad3.cu, which recomputes r1 from the inputs)
//        and the dgrad kernel (avd_dgrad3.cu)
//   MODE_CRITIC_ACTION reduces d(-mean q)/d(action) per row in the head pass itself -- the critic -> actor link
//   (trainer.py:503-506) never leaves the SM and needs no backward product at all (the V table below).
//
// BatchNorm folding (inference affine, SURVEY.md 3.3):  W2' = diag(sc1) W2,  b2' = b2 + sh1 W2  (pack_fold_kernel);
// w3' = sc2 * w3,  b3' = b3 + sh2 . w3  (table set-up below).  One CTA works on ONE agent: weights and
// tables are loaded once.  17 warps: warp 0 issues TMA / MMA, warps 1..16 are identical consumers (TMEM lane quadrant =
// warp % 4, column quarter = (warp - 1) / 4) running a software pipeline  convert(i+1) | pass2(i-1) | pass1(i)  so that
// every MMA has a full stage of other work to hide behind.
// Reference semantics: agent/model.py:19-37 (actor), 55-83 (critic); workers/trainer.py:489-506.
#include "avd_common.cuh"
#include "avd_ddpg_layout.cuh"
#include "avd_learn_kernels.cuh"
#include "avd_umma.cuh"

namespace avd {
namespace fused3 {

using namespace umma;

constexpr int TILE_M = 128, L2N = 128, KB = 64, MAX_KB = 5, L1N = 256;
constexpr int NCONS = 16;
constexpr int NUM_THREADS = 32 * (1 + NCONS);
constexpr int SLOT_BYTES = TILE_M * KB * 2;                  // 16 KB
constexpr int MAX_SLOT = 7;
constexpr int OFF_W = 0;                                     // W2'^T k-blocks
constexpr int OFF_RING = OFF_W + MAX_KB * SLOT_BYTES;        // ring of r1 k-blocks: 7 slots in the forward modes, 5 when ...
constexpr int OFF_DZ = OFF_RING + 5 * SLOT_BYTES;            // ... the last two hold the dz2 tile (2 k-blocks) of the backward modes
constexpr int OFF_B1 = OFF_RING + MAX_SLOT * SLOT_BYTES;     // W1ext, no-swizzle K-major [2 chunks][256 rows][16 B]
constexpr int B1_BYTES = 2 * L1N * 16;
constexpr int OFF_X = OFF_B1 + B1_BYTES;                     // 2 input tiles [2 chunks][128 rows][16 B]
constexpr int X_BYTES = 2 * TILE_M * 16;
constexpr int OFF_TAB = OFF_X + 2 * X_BYTES;                 // b2f[128] w3f[128] wa[64] ba[64] scal[8]
constexpr int TAB_BYTES = 2048;
constexpr int OFF_PART = OFF_TAB + TAB_BYTES;                // [2 buffers][4 quarters][128 rows] partial row sums
constexpr int OFF_BAR = OFF_PART + 2 * 4 * TILE_M * 4;
constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;
// V table of MODE_CRITIC_ACTION (in the dz2-tile slots): (la + 1) rows of 128 fp32, row pitch 132 floats so that the rows the 8 lanes
// of a quarter warp gather (one row per lane: its own action interval) spread over all bank groups; sorted breakpoints behind it
constexpr int kVRows = 49, kVStride = 132, kVBrk = 64;
static_assert((kVRows * kVStride + kVBrk) * 4 + 2 * 4 * TILE_M * 4 <= 2 * SLOT_BYTES, "V table + partial sums exceed the dz2-tile slots");
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");

struct Args {
    avd_net_dims d;
    int A;
    int64_t R;
    const float* params;        // [A][pstride]
    int64_t pstride;
    const float* b2f;           // [A][128] folded layer-2 bias
    const float* s;             // element (n, k) at s[n*s_rs + k*s_cs]
    int64_t s_rs, s_cs;
    const float* act;           // [A*R] critic passes
    const float* rew;           // MODE_TARGET
    float gamma, high;
    const float* y;             // MODE_CRITIC_BWD: TD targets
    float* out;                 // forward modes: [A*R]; MODE_CRITIC_ACTION: d loss / d action; MODE_CRITIC_BWD: q (nullable)
    uint32_t* mask_out;         // backward modes / MODE_ACTOR_SAVE: [A*R][mask_words] sign bits of z1 (column j of word w at bit 31-j)
    int mask_words;
    uint32_t* mask2_out;        // MODE_ACTOR_SAVE: [A*R][4] sign bits of z2 + b2'
    float* dact_out;            // MODE_ACTOR_SAVE: [A*R] high (1 - tanh^2(pre-activation))
    const float* vtab;          // MODE_CRITIC_ACTION: [A][kVRows][128] V table, [A][kVBrk] sorted breakpoints behind it (critic_vtab_kernel)
    float dm_scale;             // backward modes: power-of-two factor on the dm tile (1 for bf16; fp16 needs dq ~ 1 / R lifted into its range)
    float* sdq;                 // backward modes: [A]       += sum_n dq_n
    float* loss;                // nullable; element 2*agent (+1 for the actor loss)
    int tiles_per_agent, ctas_per_agent;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) {
    __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint64_t make_desc_noswz(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ void split_bf16(float v, bf16& hi, bf16& lo) {
    hi = __float2bfloat16_rn(v);
    lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack2(bf16 a, bf16 b) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// F16 (precision = 2): the layer-2 operands r1 and W2'^T and the backward tile dm are fp16 instead of bf16 (same tensor-pipe
// rate, 11-bit significand; B200 has no mixed fp16 x bf16 MMA).  dm = dq [z2 > 0] is written as dm_scale * dq with a power-of-two
// dm_scale ~ R (dq ~ 1 / R would sit in the subnormal range of fp16), saturating; the unfold kernel divides it out.
//
// MODE_CRITIC_ACTION -- d q / d action without a backward product.  The action enters the critic through ONE scalar:
//   za_f = wa_f a + ba_f,   d q / d a = sum_f [za_f > 0] wa_f sum_j [z2_j + b2'_j > 0] W2'[l1 + f][j] w3'_j          (model.py:69-83)
// As a function of a the sign pattern [za_f > 0] is piecewise constant with at most la breakpoints -ba_f / wa_f, so
//   d q / d a = sum_j [z2_j + b2'_j > 0] V[k(a)][j],     V[k][j] = sum_{f active in interval k} wa_f W2'[l1 + f][j] w3'_j,
// with k(a) = number of breakpoints below a.  critic_vtab_kernel (avd_ddpg.cu) builds the (la + 1) x 128 fp32 table and the sorted
// breakpoints per agent; the table sits in the shared memory the other backward modes use for the dz2 tile, and the head pass adds
// V[k][j] over its columns with z2_j + b2'_j > 0.  Round 1 ran the action columns of the dgrad as a third MMA on a bf16 tile
// dq w3' [z2 > 0] (a 32 KB tile written by all consumer warps per row tile, 8 MMAs, a TMEM read-back and a fourth pipeline stage:
// 160 us, and a 0.5 % bias on every actor gradient from the two bf16 roundings); this is exact in fp32.
template <int MODE, bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1) fused3_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmDZ, Args g) {
    constexpr bool CRITIC = MODE != MODE_ACTOR_OUT && MODE != MODE_ACTOR_SAVE;
    constexpr bool SAVE = MODE == MODE_ACTOR_SAVE;                               // forward pass that keeps its sign masks
    constexpr bool BWD = MODE == MODE_CRITIC_BWD;                                // full backward: masks, r1 / dz2 to HBM, U
    constexpr bool ACTION = MODE == MODE_CRITIC_ACTION;                          // forward + d q / d action (V table)
    constexpr bool HAS_DZ = BWD;
    constexpr int NKB = CRITIC ? 5 : 4;
    // k-block kb of local tile t lives in ring slot (t NKB + kb) % NSLOT: with more slots than k-blocks the converters of the
    // next tile start while the layer-2 MMA of this tile still reads its operands
    constexpr int NSLOT = (HAS_DZ || ACTION) ? 5 : MAX_SLOT;                     // the last two slots: dz2 tile (BWD) / V table (ACTION)
    constexpr uint32_t FOP = F16 ? FMT_F16 : FMT_BF16;                           // format of the layer-2 operands

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    float* b2f_tab = reinterpret_cast<float*>(smem + OFF_TAB);
    float* w3f_tab = b2f_tab + L2N;
    float* wa_tab = w3f_tab + L2N;
    float* ba_tab = wa_tab + 64;
    float* scal = ba_tab + 64;                                   // [1..4] partial sums of sh2 . w3, [5] = b3
    float* part = reinterpret_cast<float*>(smem + OFF_PART);
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + OFF_BAR);   // [7]
    uint64_t* a_empty = a_full + MAX_SLOT;                            // [7]
    uint64_t* acc_full = a_empty + MAX_SLOT;                          // [2]
    uint64_t* acc_empty = acc_full + 2;                               // [2]
    uint64_t* part_full = acc_empty + 2;                              // [2]
    uint64_t* x_full = part_full + 2;                                 // [2]
    uint64_t* z1_full = x_full + 2;
    uint64_t* z1_empty = z1_full + 1;
    uint64_t* dz_full = z1_empty + 1;
    uint64_t* dz_empty = dz_full + 1;
    uint64_t* dra_full = dz_empty + 1;
    uint64_t* dra_empty = dra_full + 1;
    uint64_t* w_full = dra_empty + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const avd_net_dims d = g.d;
    const int la = CRITIC ? d.la : 0;
    const int agent = (int)blockIdx.x / g.ctas_per_agent;
    const int cta = (int)blockIdx.x - agent * g.ctas_per_agent;
    const int T = (g.tiles_per_agent - cta + g.ctas_per_agent - 1) / g.ctas_per_agent;   // tiles of this CTA: cta, cta + ctas_per_agent, ...
    const float* P = g.params + (int64_t)agent * g.pstride;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmW);
        if (BWD) tma_prefetch_desc(&tmDZ);
        for (int i = 0; i < MAX_SLOT; ++i) { mbar_init(&a_full[i], 8); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], NCONS);
            mbar_init(&part_full[i], NCONS); mbar_init(&x_full[i], 4);
        }
        mbar_init(z1_full, 1); mbar_init(z1_empty, NCONS);
        mbar_init(dz_full, NCONS); mbar_init(dz_empty, 1);
        mbar_init(dra_full, 1); mbar_init(dra_empty, 4);
        mbar_init(w_full, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);

    // ---- per-agent tables and the extended layer-1 weight tile (built once: one CTA = one agent)
    if (warp >= 1) {
        const int ct = threadIdx.x - 32;     // 0..511
        int64_t oW, ob, og2, obe2, omu2, ovar2, oW3, ob3;
        if (CRITIC) { const CriticOff o = critic_off(d); oW = o.Ws; ob = o.bs; og2 = o.g2; obe2 = o.be2; omu2 = o.mu2; ovar2 = o.var2; oW3 = o.W3; ob3 = o.b3; }
        else { const ActorOff o = actor_off(d); oW = o.W1; ob = o.b1; og2 = o.g2; obe2 = o.be2; omu2 = o.mu2; ovar2 = o.var2; oW3 = o.W3; ob3 = o.b3; }
        if (ct < L1N) {   // W1ext row of layer-1 output column ct:  [W_hi b_hi | W_hi b_hi | W_lo b_lo | 0]  (K = 16)
            bf16 whi[4], wlo[4], bhi, blo;
#pragma unroll
            for (int k = 0; k < 4; ++k) split_bf16(k < d.ns ? P[oW + (int64_t)k * d.l1 + ct] : 0.0f, whi[k], wlo[k]);
            split_bf16(P[ob + ct], bhi, blo);
            const bf16 zero = __float2bfloat16_rn(0.0f);
            const uint4 c0 = make_uint4(pack2(whi[0], whi[1]), pack2(whi[2], whi[3]), pack2(bhi, whi[0]), pack2(whi[1], whi[2]));
            const uint4 c1 = make_uint4(pack2(whi[3], bhi), pack2(wlo[0], wlo[1]), pack2(wlo[2], wlo[3]), pack2(blo, zero));
            *reinterpret_cast<uint4*>(smem + OFF_B1 + ct * 16) = c0;
            *reinterpret_cast<uint4*>(smem + OFF_B1 + L1N * 16 + ct * 16) = c1;
        } else if (ct < L1N + L2N) {
            const int c = ct - L1N;
            const float sc2 = P[og2 + c] / sqrtf(P[ovar2 + c] + kBnEps);
            const float sh2 = P[obe2 + c] - P[omu2 + c] * sc2;
            const float w3 = P[oW3 + c];
            w3f_tab[c] = w3 * sc2;
            const float t = warp_sum(sh2 * w3);                  // four full warps hold the 128 columns
            if (lane == 0) scal[1 + (c >> 5)] = t;
            if (c == 0) scal[5] = P[ob3];
        } else if (ct < L1N + L2N + 64) {
            const int c = ct - L1N - L2N;
            float wa = 0.f, ba = 0.f;
            if (CRITIC && c < d.la) { const CriticOff o = critic_off(d); wa = P[o.Wa + c]; ba = P[o.ba + c]; }
            wa_tab[c] = wa;
            ba_tab[c] = ba;
        }
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Everything above only read the parameters (last written by the previous step's Adam / Polyak launch).  From here on the
    // kernel consumes what earlier launches of this step produced (folded weights and bias, actions, TD targets, dz2 ...).
    pdl_wait();
    pdl_launch_dependents();
    if (threadIdx.x >= 32 && threadIdx.x < 32 + L2N) b2f_tab[threadIdx.x - 32] = g.b2f[(int64_t)agent * L2N + threadIdx.x - 32];   // written by the pack kernel, possibly the previous launch
    float* vtab_s = reinterpret_cast<float*>(smem + OFF_DZ);                 // ACTION: [kVRows][kVStride] V table
    float* vbrk_s = vtab_s + kVRows * kVStride;                              //         [kVBrk] sorted breakpoints (+inf padded)
    float* part2 = vbrk_s + kVBrk;                                           //         [2 buffers][4 quarters][128 rows] partial d q / d a
    if (ACTION) {
        const float4* src = reinterpret_cast<const float4*>(g.vtab + (int64_t)agent * (kVRows * kVStride + kVBrk));
        for (int i = threadIdx.x; i < (kVRows * kVStride + kVBrk) / 4; i += NUM_THREADS) reinterpret_cast<float4*>(vtab_s)[i] = src[i];
    }
    __syncthreads();
    const float b3f = scal[5] + scal[1] + scal[2] + scal[3] + scal[4];       // b3' = b3 + sh2 . w3
    if (T <= 0) {   // never happens with the host-side grid; keep the TMEM bookkeeping correct anyway
        __syncthreads();
        if (warp == 0) tmem_dealloc(tmem_base, 512);
        return;
    }

    auto tile_of = [&](int tc) { return cta + tc * g.ctas_per_agent; };

    if (warp == 0) {
        // ============================================ TMA / MMA issuer ============================================
        // warp-uniform control flow; the one-thread instructions are predicated on an elected lane (see avd_umma.cuh)
        {
            const uint32_t leader = elect_one();
            constexpr uint32_t idesc1 = make_idesc_bf16(TILE_M, L2N, false, false);      // layer 1: hi/lo-split bf16
            constexpr uint32_t idesc = make_idesc_f16kind(TILE_M, L2N, false, false, FOP, FOP);
            const int F = L1N + la;
            const uint64_t dW = make_smem_desc(smem_u32(smem + OFF_W), 16, 1024);
            const uint64_t dR = make_smem_desc(smem_u32(smem + OFF_RING), 16, 1024);
            const uint64_t dX = make_desc_noswz(smem_u32(smem + OFF_X), TILE_M * 16, 128);
            const uint64_t dB1 = make_desc_noswz(smem_u32(smem + OFF_B1), L1N * 16, 128);
            mbar_expect_tx_p(leader, w_full, (uint32_t)NKB * SLOT_BYTES);
            for (int kb = 0; kb < NKB; ++kb) tma_load_3d_p(leader, smem + OFF_W + kb * SLOT_BYTES, &tmW, w_full, kb * KB, 0, agent);

            auto mma1 = [&](int t) {          // layer 1 of local tile t -> TMEM columns [256, 512)
                mbar_wait(&x_full[t & 1], ((uint32_t)t >> 1) & 1);
                if (t >= 1) mbar_wait(z1_empty, (uint32_t)(t - 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    mma_bf16_p(leader, tmem_base + 256u + (uint32_t)(h * L2N), desc_add(dX, (uint32_t)(t & 1) * X_BYTES), desc_add(dB1, h * (L2N * 16)), idesc1, 0);
                mma_commit_p(leader, z1_full);
            };
            auto mma2 = [&](int t) {          // layer 2 of local tile t -> TMEM accumulator t & 1
                mbar_wait(&acc_empty[t & 1], (((uint32_t)t >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)((t & 1) * L2N);
#pragma unroll
                for (int kb = 0; kb < NKB; ++kb) {
                    const uint32_t kc = (uint32_t)(t * NKB + kb), sl = kc % NSLOT;
                    mbar_wait(&a_full[sl], (kc / NSLOT) & 1);
                    tc_fence_after();
                    const int nm = min(4, (F - kb * KB) / 16);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (j < nm)
                            mma_bf16_p(leader, tacc, desc_add(dR, sl * SLOT_BYTES + j * 32), desc_add(dW, kb * SLOT_BYTES + j * 32), idesc, (kb | j) != 0);
                    mma_commit_p(leader, &a_empty[sl]);
                }
                mma_commit_p(leader, &acc_full[t & 1]);
            };
            auto dz_out = [&](int t) {        // dz2 tile of local tile t to HBM; the tile is free again once the TMA stores have read it
                mbar_wait(dz_full, (uint32_t)t & 1);
                tc_fence_after();
                tma_store_3d_p(leader, &tmDZ, smem + OFF_DZ, 0, tile_of(t) * TILE_M, agent);
                tma_store_3d_p(leader, &tmDZ, smem + OFF_DZ + SLOT_BYTES, KB, tile_of(t) * TILE_M, agent);
                if (leader) {
                    bulk_commit();
                    bulk_wait_read0();
                }
                __syncwarp();
                mbar_arrive_p(leader, dz_empty);
            };

            mbar_wait(w_full, 0);
            {
                // The tensor pipe executes in issue order: the (tiny) layer-1 MMA of the NEXT tile goes in front of the layer-2
                // MMA, so that the converters of the next iteration never wait behind a whole layer-2 product.
                mma1(0);
                if (T > 1) mma1(1);
                mma2(0);
                for (int i = 0; i < T; ++i) {
                    if (i + 1 < T) {
                        if (i + 2 < T) mma1(i + 2);
                        mma2(i + 1);
                    }
                    if (BWD && i >= 1) dz_out(i - 1);
                }
                if (BWD) dz_out(T - 1);
            }
        }
    } else {
        // ================================================ consumers ================================================
        const int cw = warp - 1;
        const int q = warp & 3;              // TMEM lane quadrant of this warp
        const int c4 = cw >> 2;              // column quarter: z1 columns [64 c4, +64), z2 columns [32 c4, +32)
        const int row = q * 32 + lane;
        const uint32_t tlane = (uint32_t)(q * 32) << 16;
        const float invR = 1.0f / (float)g.R;
        float sdq_acc = 0.0f, loss_acc = 0.0f;
        uint32_t zneg = 0u;                  // backward modes: sign bits of z2 + b2' of this thread's 32 columns (column j at bit 31 - j), pass 1 -> pass 2

        auto rowinfo = [&](int tc, bool& valid) -> int64_t {
            const int64_t r_in = (int64_t)tile_of(tc) * TILE_M + row;
            valid = r_in < g.R;
            return (int64_t)agent * g.R + (valid ? r_in : g.R - 1);
        };
        // Per-row global inputs are fetched one stage ahead of their use and carried in registers: a load issued right before
        // its use would put a full global-memory latency on the critical path of every tile.
        //   xs   : state row of the tile whose X buffer this thread's quarter writes at the end of its next convert()
        //   a_pf : action of the next tile whose action-branch columns this quarter converts
        //   y_pf : reward / TD target of the tile whose pass 2 comes next;  a_ag: action of the next pass1() (ACTION)
        float xs[4] = {0.f, 0.f, 0.f, 0.f}, a_pf = 0.0f, y_pf = 0.0f, a_ag = 0.0f;
        auto xg_of = [&](int tc) { return CRITIC ? 2 * (1 - (tc & 1)) : (tc & 3); };      // quarter that stages tile tc + 2 during convert(tc)
        auto is_action_quarter = [&](int tc) { return CRITIC && (c4 >> 1) == (tc & 1); };   // quarters 2 (tc & 1), 2 (tc & 1) + 1
        auto load_x = [&](int t) {
            bool valid;
            const int64_t n = rowinfo(t, valid);
#pragma unroll
            for (int k = 0; k < 4; ++k) xs[k] = k < d.ns ? __ldg(g.s + n * g.s_rs + k * g.s_cs) : 0.0f;
        };
        // hi/lo-split input row of local tile t -> X buffer t & 1:  [v_hi(5) v_lo(5) v_hi(5) 0],  v = (s0..s3, 1)
        auto write_x = [&](int t) {
            bf16 hi[5], lo[5];
#pragma unroll
            for (int k = 0; k < 4; ++k) split_bf16(xs[k], hi[k], lo[k]);
            hi[4] = __float2bfloat16_rn(1.0f);
            lo[4] = __float2bfloat16_rn(0.0f);
            uint8_t* xbase = smem + OFF_X + (t & 1) * X_BYTES;
            *reinterpret_cast<uint4*>(xbase + row * 16) = make_uint4(pack2(hi[0], hi[1]), pack2(hi[2], hi[3]), pack2(hi[4], lo[0]), pack2(lo[1], lo[2]));
            *reinterpret_cast<uint4*>(xbase + TILE_M * 16 + row * 16) =
                make_uint4(pack2(lo[3], lo[4]), pack2(hi[0], hi[1]), pack2(hi[2], hi[3]), pack2(hi[4], lo[4]));
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&x_full[t & 1]);
        };

        // ---- stage 1: z1 -> relu -> bf16 A tile (+ sign masks), action-branch columns, next input tile
        auto convert = [&](int tc) {
            bool valid;
            const int64_t nrow = rowinfo(tc, valid);
            const int ga0 = CRITIC ? 2 * (tc & 1) : -1;          // quarter that converts action columns 0..31; ga0 + 1: columns 32..la-1
            const float a_val = a_pf;
            mbar_wait(z1_full, (uint32_t)tc & 1);
            tc_fence_after();
            const uint32_t kc = (uint32_t)(tc * NKB + c4), sl = kc % NSLOT;
            mbar_wait(&a_empty[sl], ((kc / NSLOT) & 1) ^ 1);
            uint8_t* slot = smem + OFF_RING + sl * SLOT_BYTES + row * 128;
            uint32_t neg[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float z[32];
                tmem_ld32(tmem_base + 256u + (uint32_t)(c4 * 64 + h * 32) + tlane, z);
                uint32_t m = 0;
                if (BWD || SAVE) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) m = __funnelshift_l(__float_as_uint(z[j]), m, 1);
                }
                neg[h] = m;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint4 pk = make_uint4(pack_relu_x2<F16>(z[8 * k], z[8 * k + 1]), pack_relu_x2<F16>(z[8 * k + 2], z[8 * k + 3]),
                                                pack_relu_x2<F16>(z[8 * k + 4], z[8 * k + 5]), pack_relu_x2<F16>(z[8 * k + 6], z[8 * k + 7]));
                    *reinterpret_cast<uint4*>(slot + (((h * 4 + k) ^ (row & 7)) << 4)) = pk;      // SWIZZLE_128B
                }
            }
            tc_fence_before();
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { mbar_arrive(z1_empty); mbar_arrive_cnt(&a_full[sl], 2); }   // every slot barrier counts 8: 4 warps x 2 here, 8 warps x 1 for the action block
            if ((BWD || SAVE) && valid) *reinterpret_cast<uint2*>(g.mask_out + nrow * g.mask_words + 2 * c4) = make_uint2(neg[0], neg[1]);
            if (CRITIC && (c4 == ga0 || c4 == ga0 + 1)) {        // action branch: one input per column, CUDA cores
                const int j0 = (c4 == ga0) ? 0 : 32;
                const uint32_t kca = (uint32_t)(tc * NKB + 4), sla = kca % NSLOT;
                mbar_wait(&a_empty[sla], ((kca / NSLOT) & 1) ^ 1);
                uint8_t* aslot = smem + OFF_RING + sla * SLOT_BYTES + row * 128;
                float z[32];
                uint32_t m = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    z[j] = fmaf(a_val, wa_tab[j0 + j], ba_tab[j0 + j]);
                    if (BWD) m = __funnelshift_l(__float_as_uint(z[j]), m, 1);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int col = j0 + 8 * k;
                    if (col < la) {
                        const uint4 pk = make_uint4(pack_relu_x2<F16>(z[8 * k], z[8 * k + 1]), pack_relu_x2<F16>(z[8 * k + 2], z[8 * k + 3]),
                                                    pack_relu_x2<F16>(z[8 * k + 4], z[8 * k + 5]), pack_relu_x2<F16>(z[8 * k + 6], z[8 * k + 7]));
                        *reinterpret_cast<uint4*>(aslot + (((col >> 3) ^ (row & 7)) << 4)) = pk;
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[sla]);
                if (BWD && valid) g.mask_out[nrow * g.mask_words + 8 + (j0 >> 5)] = m;
            }
            if (c4 == xg_of(tc) && tc + 2 < T) write_x(tc + 2);  // X buffer tc & 1 is free: z1_full(tc) implies the layer-1 MMA has read it
            // prefetch for the next convert()
            if (tc + 3 < T && c4 == xg_of(tc + 1)) load_x(tc + 3);
            if (tc + 1 < T && is_action_quarter(tc + 1)) {
                bool v1;
                a_pf = __ldg(g.act + rowinfo(tc + 1, v1));
            }
        };

        // ---- stage 2: partial row sums of the head over this warp's 32 z2 columns
        auto pass1 = [&](int tc) {
            const int buf = tc & 1;
            if (MODE == MODE_TARGET || BWD) {                    // consumed by pass2(tc), one iteration later
                bool v0;
                const int64_t n0 = rowinfo(tc, v0);
                if (MODE == MODE_TARGET) { if (c4 == 0) y_pf = __ldg(g.rew + n0); }
                else y_pf = __ldg(g.y + n0);
            }
            const float* vrow = vtab_s;          // ACTION: this row's V[k(a)] (its 32 columns), k(a) = breakpoints below the action
            if (ACTION) {
                const float a_cur = a_ag;
                if (tc + 1 < T) {
                    bool v1;
                    a_ag = __ldg(g.act + rowinfo(tc + 1, v1));
                }
                int k = 0;
#pragma unroll
                for (int st = 32; st >= 1; st >>= 1)
                    if (vbrk_s[k + st - 1] < a_cur) k += st;
                vrow = vtab_s + k * kVStride + c4 * 32;
            }
            mbar_wait(&acc_full[buf], ((uint32_t)tc >> 1) & 1);
            tc_fence_after();
            float v[32];
            tmem_ld32(tmem_base + (uint32_t)(buf * L2N + c4 * 32) + tlane, v);
            float acc = 0.0f, gacc = 0.0f;
            uint32_t m = 0u;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(b2f_tab + c4 * 32 + j);
                const float4 w4 = *reinterpret_cast<const float4*>(w3f_tab + c4 * 32 + j);
                const float t0 = v[j] + b4.x, t1 = v[j + 1] + b4.y, t2 = v[j + 2] + b4.z, t3 = v[j + 3] + b4.w;
                if (ACTION) {        // + V[k][j] where z2_j + b2'_j > 0 (sign bit clear): AND with the inverted sign mask, no branch
                    const float4 V4 = *reinterpret_cast<const float4*>(vrow + j);
                    gacc += __uint_as_float(__float_as_uint(V4.x) & ~(uint32_t)((int32_t)__float_as_uint(t0) >> 31));
                    gacc += __uint_as_float(__float_as_uint(V4.y) & ~(uint32_t)((int32_t)__float_as_uint(t1) >> 31));
                    gacc += __uint_as_float(__float_as_uint(V4.z) & ~(uint32_t)((int32_t)__float_as_uint(t2) >> 31));
                    gacc += __uint_as_float(__float_as_uint(V4.w) & ~(uint32_t)((int32_t)__float_as_uint(t3) >> 31));
                }
                acc = fmaf(fmaxf(t0, 0.0f), w4.x, acc);
                acc = fmaf(fmaxf(t1, 0.0f), w4.y, acc);
                acc = fmaf(fmaxf(t2, 0.0f), w4.z, acc);
                acc = fmaf(fmaxf(t3, 0.0f), w4.w, acc);
                if (HAS_DZ || SAVE) {
                    m = __funnelshift_l(__float_as_uint(t0), m, 1);
                    m = __funnelshift_l(__float_as_uint(t1), m, 1);
                    m = __funnelshift_l(__float_as_uint(t2), m, 1);
                    m = __funnelshift_l(__float_as_uint(t3), m, 1);
                }
            }
            if (HAS_DZ) zneg = m;
            if (SAVE) {
                bool v1;
                const int64_t n1 = rowinfo(tc, v1);
                if (v1) g.mask2_out[n1 * 4 + c4] = m;
            }
            part[(buf * 4 + c4) * TILE_M + row] = acc;
            if (ACTION) part2[(buf * 4 + c4) * TILE_M + row] = gacc;
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                // Pass 2 of the backward modes works from the sign bits kept above, so the accumulator is free again.  In the forward
                // modes the quarter-0 warps release it in pass 2 instead: the layer-2 MMA of tile tc + 2 (and with it every
                // pass1(tc + 2) that overwrites `part`) then cannot start before they have combined the partial sums of tile tc.
                if (HAS_DZ || c4 != 0) mbar_arrive(&acc_empty[buf]);
                mbar_arrive(&part_full[buf]);
            }
        };

        // ---- stage 3: combine the row sums; outputs; backward modes: dq, dz2 tile, U / loss accumulation
        auto pass2 = [&](int tc) {
            const int buf = tc & 1;
            if (!HAS_DZ && c4 != 0) return;
            bool valid;
            const int64_t nrow = rowinfo(tc, valid);
            const float yv = y_pf;
            mbar_wait(&part_full[buf], ((uint32_t)tc >> 1) & 1);
            const float* pb = part + buf * 4 * TILE_M + row;
            const float qv = pb[0] + pb[TILE_M] + pb[2 * TILE_M] + pb[3 * TILE_M] + b3f;
            if (!HAS_DZ) {
                float o;
                if (MODE == MODE_ACTOR_OUT || SAVE) {
                    const float t = tanhf(qv);
                    o = g.high * t;
                    if (SAVE && valid) g.dact_out[nrow] = g.high * (1.0f - t * t);       // through high * tanh(.)    model.py:36-37
                }
                else if (MODE == MODE_TARGET) o = yv + g.gamma * qv;                 // trainer.py:494 (no terminal mask)
                else if (ACTION) {                                                   // d(-mean q)/d a   trainer.py:503-506
                    const float* pg = part2 + buf * 4 * TILE_M + row;
                    o = -invR * (pg[0] + pg[TILE_M] + pg[2 * TILE_M] + pg[3 * TILE_M]);
                    if (valid) loss_acc -= qv * invR;                                // -mean q          trainer.py:504
                }
                else o = qv;
                if (valid) g.out[nrow] = o;
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
                return;
            }
            const float diff = qv - yv;
            const float dq = valid ? 2.0f * diff * invR : 0.0f;                      // d mean((y-q)^2) / dq      trainer.py:496
            if (c4 == 0) {
                if (valid) loss_acc = fmaf(diff, diff * invR, loss_acc);
                if (valid && g.out) g.out[nrow] = qv;
            }
            if (c4 == 0) sdq_acc += dq;
            float v[32];
            {
                // The tile holds dq [z2 + b2' > 0] WITHOUT the head weight w3': it is folded into the dgrad operand (W2'' = W2' diag(w3'),
                // pack_fold4_kernel) and into the unfold of the weight gradient, where U = sum_n dq_n relu(z2 + b2') also comes out
                // of G2 (sum_f W2'[f][j] G2[f][j] + b2'[j] db2[j]) instead of 32 accumulator registers per thread here.  The sign
                // bits come from pass 1, so the TMEM accumulator was released a whole stage earlier.
                const float dqs = dq * g.dm_scale;
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = (zneg & (0x80000000u >> j)) ? 0.0f : dqs;
            }
            mbar_wait(dz_empty, ((uint32_t)tc & 1) ^ 1);
            uint8_t* dzrow = smem + OFF_DZ + (c4 >> 1) * SLOT_BYTES + row * 128;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint4 pk = make_uint4(pack_x2<F16>(v[8 * k], v[8 * k + 1]), pack_x2<F16>(v[8 * k + 2], v[8 * k + 3]),
                                            pack_x2<F16>(v[8 * k + 4], v[8 * k + 5]), pack_x2<F16>(v[8 * k + 6], v[8 * k + 7]));
                *reinterpret_cast<uint4*>(dzrow + ((((c4 & 1) * 4 + k) ^ (row & 7)) << 4)) = pk;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(dz_full);
        };

        // ---- software pipeline
        if (cw < 4) { load_x(0); write_x(0); }
        else if (cw < 8 && T > 1) { load_x(1); write_x(1); }
        if (T > 2 && c4 == xg_of(0)) load_x(2);
        if (is_action_quarter(0)) {
            bool v0;
            a_pf = __ldg(g.act + rowinfo(0, v0));
        }
        if (ACTION) {
            bool v0;
            a_ag = __ldg(g.act + rowinfo(0, v0));
        }
        convert(0);
        for (int i = 0; i < T; ++i) {
            {                                // every stage waits on work that is at least one stage old
                if (i + 1 < T) convert(i + 1);
                if (i >= 1) pass2(i - 1);
                pass1(i);
            }
        }
        pass2(T - 1);

        // ---- flush the per-thread partial sums of this CTA
        if ((HAS_DZ || ACTION) && c4 == 0) {
            const float sl = warp_sum(loss_acc), sd = warp_sum(sdq_acc);
            if (lane == 0) {
                if (g.loss) atomicAdd(g.loss + 2 * agent + (MODE == MODE_CRITIC_BWD ? 0 : 1), sl);
                if (BWD) atomicAdd(g.sdq + agent, sd);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

bool supported(const avd_net_dims& d) {       // la <= 48: the V table of the critic-action pass has la + 1 <= kVRows rows
    return d.l2 == L2N && d.ns >= 1 && d.ns <= 4 && d.l1 == L1N && d.la % 16 == 0 && d.la >= 16 && d.la < kVRows;
}
int vtab_rows() { return kVRows; }
int vtab_stride() { return kVStride; }
int vtab_floats() { return kVRows * kVStride + kVBrk; }

template <int MODE, bool F16>
static int launch2(const CUtensorMap& tmW, const CUtensorMap& tmDZ, const Args& g, dim3 grid, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        AVD_CUDA_OK(cudaFuncSetAttribute(fused3_kernel<MODE, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    AVD_CUDA_OK(launch_pdl(fused3_kernel<MODE, F16>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tmW, tmDZ, g));
    AVD_LAUNCH_OK();
    return AVD_OK;
}
template <int MODE>
static int launch(bool f16, const CUtensorMap& tmW, const CUtensorMap& tmDZ, const Args& g, dim3 grid, cudaStream_t st) {
    return f16 ? launch2<MODE, true>(tmW, tmDZ, g, grid, st) : launch2<MODE, false>(tmW, tmDZ, g, grid, st);
}

// One pass (the buffers are described at RunArgs, avd_learn_kernels.cuh).
int run(const RunArgs& a, cudaStream_t st) {
    const avd_net_dims& d = a.d;
    if (!supported(d)) {
        set_error("fused pass kernel does not support these layer sizes");
        return AVD_ERR_UNSUPPORTED;
    }
    const int mode = a.mode;
    const bool critic = mode != MODE_ACTOR_OUT && mode != MODE_ACTOR_SAVE;
    const bool bwd = mode == MODE_CRITIC_BWD;
    const int F = critic ? d.l1 + d.la : d.l1;
    AVD_REQUIRE(a.params && a.W2T && a.b2f && a.s, "null buffer");
    AVD_REQUIRE(a.A >= 1 && a.R >= 1 && a.R < (int64_t)1 << 31, "rows per agent must fit the 32-bit TMA coordinates");
    AVD_REQUIRE(!critic || a.act, "critic passes need actions");
    AVD_REQUIRE(!bwd || (a.mask_out && a.DZ_out && a.sdq), "backward passes need mask / dz2 / sdq outputs");
    AVD_REQUIRE(mode != MODE_CRITIC_ACTION || (a.vtab && d.la < kVRows), "the critic-action pass needs its V table (la <= %d)", kVRows - 1);
    AVD_REQUIRE(bwd || a.out, "null output");
    AVD_REQUIRE(mode != MODE_ACTOR_SAVE || (a.mask_out && a.mask2_out && a.dact_out), "MODE_ACTOR_SAVE needs the mask / d(action) outputs");
    const int A = a.A;
    const int64_t R = a.R;
    CUtensorMap tmW, tmDZ;
    if (int rc = make_tensor_map(&tmW, a.W2T, (uint64_t)F, L2N, (uint64_t)A, (uint64_t)F, (uint64_t)F * L2N, KB, TILE_M)) return rc;
    tmDZ = tmW;
    if (bwd)
        if (int rc = make_tensor_map(&tmDZ, a.DZ_out, L2N, (uint64_t)R, (uint64_t)A, L2N, (uint64_t)R * L2N, KB, TILE_M)) return rc;
    Args g;
    g.d = d; g.A = A; g.R = R; g.params = a.params; g.pstride = a.pstride; g.b2f = a.b2f; g.s = a.s; g.s_rs = a.s_rs; g.s_cs = a.s_cs; g.act = a.act;
    g.rew = a.rew; g.gamma = a.gamma; g.high = a.high; g.y = a.y; g.out = a.out; g.mask_out = a.mask_out; g.mask_words = 2 * ((F + KB - 1) / KB);
    g.vtab = a.vtab; g.dm_scale = a.dm_scale; g.sdq = a.sdq; g.loss = a.loss; g.mask2_out = a.mask2_out; g.dact_out = a.dact_out;
    g.tiles_per_agent = (int)((R + TILE_M - 1) / TILE_M);
    g.ctas_per_agent = ctas_per_agent(A, R);
    const dim3 grid((unsigned)(g.ctas_per_agent * A));
    const bool f16 = a.f16;
    switch (mode) {
        case MODE_ACTOR_OUT: return launch<MODE_ACTOR_OUT>(f16, tmW, tmDZ, g, grid, st);
        case MODE_TARGET: return launch<MODE_TARGET>(f16, tmW, tmDZ, g, grid, st);
        case MODE_Q: return launch<MODE_Q>(f16, tmW, tmDZ, g, grid, st);
        case MODE_CRITIC_BWD: return launch<MODE_CRITIC_BWD>(f16, tmW, tmDZ, g, grid, st);
        case MODE_CRITIC_ACTION: return launch<MODE_CRITIC_ACTION>(f16, tmW, tmDZ, g, grid, st);
        case MODE_ACTOR_SAVE: return launch<MODE_ACTOR_SAVE>(f16, tmW, tmDZ, g, grid, st);
    }
    set_error("unknown fused pass mode %d", mode);
    return AVD_ERR_INVALID_ARG;
}

}  // namespace fused3
}  // namespace avd
