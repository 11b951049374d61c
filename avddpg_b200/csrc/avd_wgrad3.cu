// avd_wgrad3.cu -- layer-2 weight gradient of the DDPG learn step with the activations RECOMPUTED on chip (sm_100a):
//
//   G2[f][j] += sum_n r1[n][f] dz2[n][j],      r1 = relu(x W1 + b1)   (the BN-folded formulation of avd_fused3.cu)
//
// r1 is 608 B per row as bf16; the inputs it is made of are 16-20 B.  So instead of streaming r1 back from HBM, each CTA
// loads a 128-row dz2 tile ONCE (TMA) and walks the 128-feature slabs of the layer:
//   x tile --tcgen05.mma (hi/lo split bf16, K = 16)--> z1 slab in TMEM --converter warps: relu, bf16--> r1 slab in shared
//   memory, laid out as the MN-major A operand (M = features, K = rows) --tcgen05.mma against the dz2 tile (MN-major B)-->
//   one 128 x 128 fp32 accumulator per slab; the 2-3 accumulators stay in TMEM for the whole kernel and are stored to the
//   CTA's own partial slice once at the end (the unfold kernel adds the slices up).
// HBM traffic per row: 256 B (dz2) + 16-20 B inputs; nothing is written.
// The action-branch slab of the critic (one input per feature, model.py:69-70) is converted on the CUDA cores.
// Reference: workers/trainer.py:498, 506 (tape.gradient) through agent/model.py:19-33, 62-77.
//
// Warps: 0 issuer of the G2 products, 1 TMA producer, 2..17 converters in four TEAMS of four warps (one warp per TMEM lane
// quadrant), 18 issuer of the layer-1 MMAs.  Team k owns the 64-feature unit k of every row tile (features [64 k, 64 k + 64)):
// per tile a warp waits for ONE layer-1 product, pulls its 64 values into registers (two tcgen05.ld in flight), hands the ring
// entry back at once and converts from registers -- four independent unit pipelines per CTA instead of two groups that walked the
// units of a tile one after the other (round 2, first version: 1560 cycles per unit chain against 512 cycles of tensor-pipe
// work per slab).  The action-branch features of the critic are spread over two teams, alternating with the tile parity.
// TMEM: the accumulator is G2^T -- lane = layer-2 unit j, column = feature f (the dz2 tile is the MN-major A operand, the r1 slab
// the MN-major B operand) -- 256 columns for the state features + 64 for the action branch (N = 64 products instead of a third
// 128-wide slab), which leaves a ring of four (actor) / three (critic) 64-column z1 entries.
#include "avd_common.cuh"
#include "avd_ddpg_layout.cuh"
#include "avd_learn_kernels.cuh"
#include "avd_umma.cuh"

namespace avd {
namespace wgrad3 {

using namespace umma;

constexpr int TILE_M = 128, L2N = 128, KB = 64, SLAB = 128;
constexpr int NCONV = 16;                                   // converter warps: four teams of four (one per TMEM lane quadrant), 64 columns each
constexpr int NUM_THREADS = 32 * (3 + NCONV);
constexpr int WARP_L1 = 2 + NCONV;                           // issuer of the layer-1 MMAs
constexpr int HALF_BYTES = TILE_M * 128;                     // [128 rows][64 bf16]: 16 KB
constexpr int OFF_DZ = 0;                                    // 2 x dz2 tile (2 halves of 64 columns)
constexpr int OFF_R1 = OFF_DZ + 2 * 2 * HALF_BYTES;          // 2 x r1 slab (2 halves of 64 features)
constexpr int L1N = 256;
constexpr int NRB = 4;                                       // ring of r1 slabs: deep enough that the barrier round trips converter -> issuer ->
                                                             // tensor pipe -> converter of one slab hide behind the products of the others
constexpr int OFF_B1 = OFF_R1 + NRB * 2 * HALF_BYTES;          // W1ext, no-swizzle K-major [2 chunks][256 rows][16 B]
constexpr int OFF_X = OFF_B1 + 2 * L1N * 16;                 // 2 input tiles [2 chunks][128 rows][16 B]
constexpr int X_BYTES = 2 * TILE_M * 16;
constexpr int OFF_TAB = OFF_X + 2 * X_BYTES;                 // wa[64] ba[64]
constexpr int OFF_BAR = OFF_TAB + 512;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;

struct Args {
    avd_net_dims d;
    int critic, A, FT;          // FT slab steps per row tile (actor 2; critic 3, the last one = action branch)
    int64_t R;
    const float* params;        // [A][pstride]
    int64_t pstride;
    const float* s;             // [A*R][s_rs]: the first ns words of a row
    int64_t s_rs;
    const float* act;           // [A*R] (critic)
    float* out;                 // G2 slice of CTA (agent, cta): out + agent*out_agent_stride + cta*out_cta_stride, row-major [F][128]
    int64_t out_agent_stride, out_cta_stride;
    int tiles_per_agent, ctas_per_agent;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
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

// F16 (precision = 2): the recomputed r1 slab is fp16, exactly the values the forward pass multiplied (the unfold kernel derives
// the head-weight sum U from G2, which only holds if both see the same r1), and so is the dz2 tile the backward pass wrote.
template <bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1) wgrad3_kernel(const __grid_constant__ CUtensorMap tmDZ, Args g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    float* wa_tab = reinterpret_cast<float*>(smem + OFF_TAB);
    float* ba_tab = wa_tab + 64;
    uint64_t* dz_full = reinterpret_cast<uint64_t*>(smem + OFF_BAR);  // [2]
    uint64_t* dz_empty = dz_full + 2;                                 // [2]
    uint64_t* r_full = dz_empty + 2;                                  // [NRB]
    uint64_t* r_empty = r_full + NRB;                                 // [NRB]
    uint64_t* x_full = r_empty + NRB;                                   // [2]
    uint64_t* z1_full = x_full + 2;                                   // [4]
    uint64_t* z1_empty = z1_full + 4;                                 // [4]
    uint64_t* acc_done = z1_empty + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const avd_net_dims d = g.d;
    const int agent = (int)blockIdx.x / g.ctas_per_agent;
    const int cta = (int)blockIdx.x - agent * g.ctas_per_agent;
    const int T = (g.tiles_per_agent - cta + g.ctas_per_agent - 1) / g.ctas_per_agent;
    const int FT = g.FT;                                     // slab steps per row tile: 2 state slabs (+ the action-branch step of the critic)
    const float* P = g.params + (int64_t)agent * g.pstride;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmDZ);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&dz_full[i], 1); mbar_init(&dz_empty[i], 1);
            mbar_init(&x_full[i], 4);
        }
        for (int i = 0; i < 4; ++i) { mbar_init(&z1_full[i], 1); mbar_init(&z1_empty[i], 4); }
        for (int i = 0; i < NRB; ++i) { mbar_init(&r_full[i], NCONV / 2); mbar_init(&r_empty[i], 1); }    // every step is filled by two teams
        mbar_init(acc_done, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (warp >= 2 && warp < WARP_L1) {
        const int ct = threadIdx.x - 64;     // 0..511; the first 256 build the W1ext row of layer-1 output column ct
        if (ct < L1N) {
            const int64_t oW = g.critic ? critic_off(d).Ws : actor_off(d).W1, ob = g.critic ? critic_off(d).bs : actor_off(d).b1;
            bf16 whi[4], wlo[4], bhi, blo;
#pragma unroll
            for (int k = 0; k < 4; ++k) split_bf16(k < d.ns ? P[oW + (int64_t)k * d.l1 + ct] : 0.0f, whi[k], wlo[k]);
            split_bf16(P[ob + ct], bhi, blo);
            const bf16 zero = __float2bfloat16_rn(0.0f);
            *reinterpret_cast<uint4*>(smem + OFF_B1 + ct * 16) = make_uint4(pack2(whi[0], whi[1]), pack2(whi[2], whi[3]), pack2(bhi, whi[0]), pack2(whi[1], whi[2]));
            *reinterpret_cast<uint4*>(smem + OFF_B1 + L1N * 16 + ct * 16) = make_uint4(pack2(whi[3], bhi), pack2(wlo[0], wlo[1]), pack2(wlo[2], wlo[3]), pack2(blo, zero));
        }
        if (g.critic && ct < 64) {           // zero weights beyond la: those features convert to relu(0) = 0
            const CriticOff o = critic_off(d);
            wa_tab[ct] = ct < d.la ? P[o.Wa + ct] : 0.0f;
            ba_tab[ct] = ct < d.la ? P[o.ba + ct] : 0.0f;
        }
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                      // the prologue only read the parameters; dz2 comes from the previous launch
    pdl_launch_dependents();
    auto tile_of = [&](int tc) { return cta + tc * g.ctas_per_agent; };
    // Row tile t: units u = 4 t + k (64 state features each, z1 ring entry u % NZ), slab steps q = t FT + sl (r1 buffer q % NRB):
    // sl < 2 the 128-feature state slabs (units 2 sl, 2 sl + 1), sl = 2 the action branch (64 feature columns, la of them non-zero).
    const int NZ = FT > 2 ? 3 : 4;
    const uint32_t kActCol = 2 * SLAB;                               // accumulator columns of the action-branch features
    const uint32_t zbase = tmem_base + (FT > 2 ? kActCol + 64u : kActCol);
    const int U = 4 * T;

    if (warp == 0) {
        // ================================================ MMA issuer ================================================
        // warp-uniform control flow; the tcgen05 instructions are predicated on one elected lane (see avd_umma.cuh)
        if (T > 0) {
            const uint32_t leader = elect_one();
            constexpr uint32_t FOP = F16 ? FMT_F16 : FMT_BF16;
            constexpr uint32_t idesc2 = make_idesc_f16kind(L2N, SLAB, true, true, FOP, FOP);    // dz2 tile^T (MN-major A) x r1 slab (MN-major B)
            constexpr uint32_t idesc2a = make_idesc_f16kind(L2N, 64, true, true, FOP, FOP);     // ... x the 64 action-branch columns
            const uint64_t dR = make_smem_desc(smem_u32(smem + OFF_R1), HALF_BYTES, 1024);
            const uint64_t dDZ = make_smem_desc(smem_u32(smem + OFF_DZ), HALF_BYTES, 1024);
            for (int t = 0; t < T; ++t) {
                for (int sl = 0; sl < FT; ++sl) {
                    const uint32_t q = (uint32_t)(t * FT + sl);
                    mbar_wait(&r_full[q % NRB], (q / NRB) & 1);             // converters are done with this step
                    if (sl == 0) mbar_wait(&dz_full[t & 1], ((uint32_t)t >> 1) & 1);
                    tc_fence_after();
                    const uint32_t off = (q % NRB) * 2 * HALF_BYTES, doff = (uint32_t)(t & 1) * 2 * HALF_BYTES;
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        mma_bf16_p(leader, tmem_base + (uint32_t)(sl * SLAB), desc_add(dDZ, doff + ks * 2048), desc_add(dR, off + ks * 2048), sl < 2 ? idesc2 : idesc2a,
                                   (t | ks) != 0);
                    mma_commit_p(leader, &r_empty[q % NRB]);
                    if (sl == FT - 1) mma_commit_p(leader, &dz_empty[t & 1]);
                }
            }
            mma_commit_p(leader, acc_done);
        }
    } else if (warp == WARP_L1) {
        // ============================================ layer-1 MMA issuer ============================================
        // A warp of its own: every tcgen05.commit costs the issuing thread ~140 cycles and an MMA issue blocks while the tensor
        // pipe's queue is full, so one thread issuing both products was the bottleneck of the whole kernel.
        if (T > 0) {
            const uint32_t leader = elect_one();
            const uint64_t dX = make_desc_noswz(smem_u32(smem + OFF_X), TILE_M * 16, 128);
            const uint64_t dB1 = make_desc_noswz(smem_u32(smem + OFF_B1), L1N * 16, 128);
            constexpr uint32_t idesc1h = make_idesc_bf16(TILE_M, 64, false, false);    // x (K-major) x W1ext unit (K-major)
            // The ring barriers are per TEAM (z1_full[k] / z1_empty[k]: unit k of every tile), not per ring entry: with three entries an
            // entry changes hands between teams, and a team waiting for the entry's NEXT phase while another team's phase is still
            // open would see the parity of an already completed phase.  Unit u goes into entry u % NZ, once the team of the entry's
            // previous unit u - NZ has pulled that one into registers.
            int e = 0;
            for (int u = 0; u < U; ++u) {
                const int t = u >> 2;
                if ((u & 3) == 0) mbar_wait(&x_full[t & 1], ((uint32_t)t >> 1) & 1);
                if (u >= NZ) mbar_wait(&z1_empty[(u - NZ) & 3], ((uint32_t)(u - NZ) >> 2) & 1);
                tc_fence_after();
                mma_bf16_p(leader, zbase + (uint32_t)(e * 64), desc_add(dX, (uint32_t)(t & 1) * X_BYTES), desc_add(dB1, (uint32_t)(u & 3) * 64 * 16), idesc1h, 0);
                mma_commit_p(leader, &z1_full[u & 3]);
                if (++e == NZ) e = 0;
            }
        }
    } else if (warp == 1) {
        // ================================================ TMA producer ================================================
        {
            const uint32_t leader = elect_one();
            constexpr int PF = 3;            // dz2 tiles are pulled into L2 this many tiles ahead of their shared-memory load
            for (int t = 2; t < 2 + PF && t < T; ++t) {
                tma_prefetch_3d_p(leader, &tmDZ, 0, tile_of(t) * TILE_M, agent);
                tma_prefetch_3d_p(leader, &tmDZ, KB, tile_of(t) * TILE_M, agent);
            }
            for (int t = 0; t < T; ++t) {
                const int b = t & 1;
                if (t >= 2 && t + PF < T) {
                    tma_prefetch_3d_p(leader, &tmDZ, 0, tile_of(t + PF) * TILE_M, agent);
                    tma_prefetch_3d_p(leader, &tmDZ, KB, tile_of(t + PF) * TILE_M, agent);
                }
                mbar_wait(&dz_empty[b], (((uint32_t)t >> 1) & 1) ^ 1);
                uint8_t* dst = smem + OFF_DZ + b * 2 * HALF_BYTES;
                mbar_expect_tx_p(leader, &dz_full[b], 2 * HALF_BYTES);
                tma_load_3d_p(leader, dst, &tmDZ, &dz_full[b], 0, tile_of(t) * TILE_M, agent);
                tma_load_3d_p(leader, dst + HALF_BYTES, &tmDZ, &dz_full[b], KB, tile_of(t) * TILE_M, agent);
            }
        }
    } else {
        // ================================================ converters ================================================
        const int cw = warp - 2;             // 0..15
        const int q4 = warp & 3, team = cw >> 2;     // TMEM lane quadrant; team = 64-feature unit of every tile
        const int sl_own = team >> 1, half = team & 1;
        const int row = q4 * 32 + lane;
        const uint32_t tlane = (uint32_t)(q4 * 32) << 16;
        auto rowidx = [&](int tc) -> int64_t {
            const int64_t r_in = (int64_t)tile_of(tc) * TILE_M + row;
            return (int64_t)agent * g.R + (r_in < g.R ? r_in : g.R - 1);
        };
        // Per-row inputs are fetched one tile ahead of their use (xs: state row of the tile whose X buffer is written next,
        // a_nx: action of the next tile this team converts): a load issued right before its use would put a global-memory latency on every tile.
        float xs[4] = {0.f, 0.f, 0.f, 0.f}, a_nx = 0.0f;
        auto load_x = [&](int t) {
            const int64_t n = rowidx(t);
#pragma unroll
            for (int k = 0; k < 4; ++k) xs[k] = k < d.ns ? __ldg(g.s + n * g.s_rs + k) : 0.0f;
        };
        auto write_x = [&](int t) {           // [v_hi(5) v_lo(5) v_hi(5) 0],  v = (s0..s3, 1)
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
        // the action-branch step of tile t belongs to the two teams of slab t & 1 (32 feature columns per warp)
        auto has_action = [&](int t) { return FT > 2 && sl_own == (t & 1); };
        if (team == 3 && T > 0) {         // team 3 owns the LAST unit of a tile: its z1_full means all four layer-1 MMAs have read the X buffer
            load_x(0);
            write_x(0);
            if (T > 1) { load_x(1); write_x(1); }
            if (T > 2) load_x(2);
        }
        if (T > 0 && has_action(0)) a_nx = __ldg(g.act + rowidx(0));
        int e = team % NZ;                    // ring entry (4 t + team) % NZ
        for (int t = 0; t < T; ++t) {
            float z[64];
            mbar_wait(&z1_full[team], (uint32_t)t & 1);
            tc_fence_after();
            tmem_ld64(zbase + (uint32_t)(e * 64) + tlane, z);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&z1_empty[team]);         // the values are in registers: the ring entry can be refilled
            e += 4 - NZ;
            if (e >= NZ) e -= NZ;
            const float a_val = a_nx;
            if (t + 1 < T && has_action(t + 1)) a_nx = __ldg(g.act + rowidx(t + 1));
            if (team == 3 && t + 2 < T) {                         // X buffer t & 1 is free (see above)
                write_x(t + 2);
                if (t + 3 < T) load_x(t + 3);
            }
            // rows past the end of the agent's batch: dz2 is zero-filled by TMA there, so whatever r1 holds contributes nothing
            {
                const uint32_t q = (uint32_t)(t * FT + sl_own), rb = q % NRB;
                uint8_t* rrow = smem + OFF_R1 + rb * 2 * HALF_BYTES + half * HALF_BYTES + row * 128;
                mbar_wait(&r_empty[rb], ((q / NRB) & 1) ^ 1);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint4 pk = make_uint4(pack_relu_x2<F16>(z[8 * k], z[8 * k + 1]), pack_relu_x2<F16>(z[8 * k + 2], z[8 * k + 3]),
                                                pack_relu_x2<F16>(z[8 * k + 4], z[8 * k + 5]), pack_relu_x2<F16>(z[8 * k + 6], z[8 * k + 7]));
                    *reinterpret_cast<uint4*>(rrow + ((k ^ (row & 7)) << 4)) = pk;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&r_full[rb]);
            }
            if (has_action(t)) {             // action-branch columns [32 half, +32) of the critic: one input per feature, CUDA cores
                const uint32_t q = (uint32_t)(t * FT + 2), rb = q % NRB;
                uint8_t* rrow = smem + OFF_R1 + rb * 2 * HALF_BYTES + row * 128;
                mbar_wait(&r_empty[rb], ((q / NRB) & 1) ^ 1);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float r[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) r[j] = fmaf(a_val, wa_tab[half * 32 + 8 * k + j], ba_tab[half * 32 + 8 * k + j]);
                    *reinterpret_cast<uint4*>(rrow + (((half * 4 + k) ^ (row & 7)) << 4)) =
                        make_uint4(pack_relu_x2<F16>(r[0], r[1]), pack_relu_x2<F16>(r[2], r[3]), pack_relu_x2<F16>(r[4], r[5]), pack_relu_x2<F16>(r[6], r[7]));
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&r_full[rb]);
            }
        }
        // ---- accumulator G2^T of this CTA -> global: lane = layer-2 unit j, this team's feature columns; 32 lanes write 128 contiguous bytes
        if (T > 0) {
            mbar_wait(acc_done, 0);
            tc_fence_after();
            float* dst = g.out + (int64_t)agent * g.out_agent_stride + (int64_t)cta * g.out_cta_stride + row;
            float v[64];
            tmem_ld64(tmem_base + (uint32_t)(team * 64) + tlane, v);
#pragma unroll
            for (int i = 0; i < 64; ++i) dst[(int64_t)(team * 64 + i) * L2N] = v[i];
            if (FT > 2) {
                float w[16];
                tmem_ld16(tmem_base + kActCol + (uint32_t)(team * 16) + tlane, w);
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (team * 16 + i < d.la) dst[(int64_t)(2 * SLAB + team * 16 + i) * L2N] = w[i];
            }
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

// out: every CTA (agent, cta) stores its partial G2 (row-major [F][128] fp32, rows < F) at out + agent*out_agent_stride +
// cta*out_cta_stride -- no atomics: the 37 x 4 CTAs of the C2 case would otherwise serialise 7 M atomic adds on 160 k
// addresses (a quarter of the kernel time).  The caller sums the ctas_per_agent(A, R) slices.  DZ: bf16 [A*R][128].
int run(bool f16, const avd_net_dims& d, bool critic, int A, int64_t R, const float* params, int64_t pstride, const float* s, int64_t s_rs, const float* act, const bf16* DZ,
        float* out, int64_t out_agent_stride, int64_t out_cta_stride, cudaStream_t st) {
    AVD_REQUIRE(d.l1 == 256 && d.l2 == L2N && d.ns >= 1 && d.ns <= 4 && (!critic || (d.la >= 8 && d.la <= 64)), "unsupported layer sizes for the fused wgrad kernel");
    AVD_REQUIRE(params && s && DZ && out && (!critic || act), "null buffer");
    AVD_REQUIRE(out_agent_stride % 4 == 0 && out_cta_stride % 4 == 0 && ((uintptr_t)out & 15) == 0, "partial G2 slices must be 16-byte aligned");
    static bool attr_set = false;
    if (!attr_set) {
        AVD_CUDA_OK(cudaFuncSetAttribute(wgrad3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        AVD_CUDA_OK(cudaFuncSetAttribute(wgrad3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    CUtensorMap tm;
    if (int rc = make_tensor_map(&tm, DZ, L2N, (uint64_t)R, (uint64_t)A, L2N, (uint64_t)R * L2N, KB, TILE_M)) return rc;
    Args g;
    g.d = d; g.critic = critic ? 1 : 0; g.A = A; g.FT = critic ? 3 : 2; g.R = R; g.params = params; g.pstride = pstride; g.s = s; g.s_rs = s_rs; g.act = act;
    g.out = out; g.out_agent_stride = out_agent_stride; g.out_cta_stride = out_cta_stride;
    g.tiles_per_agent = (int)((R + TILE_M - 1) / TILE_M);
    g.ctas_per_agent = ctas_per_agent(A, R);
    if (f16) AVD_CUDA_OK(launch_pdl(wgrad3_kernel<true>, dim3((unsigned)(A * g.ctas_per_agent)), dim3(NUM_THREADS), SMEM_BYTES, st, tm, g));
    else AVD_CUDA_OK(launch_pdl(wgrad3_kernel<false>, dim3((unsigned)(A * g.ctas_per_agent)), dim3(NUM_THREADS), SMEM_BYTES, st, tm, g));
    AVD_LAUNCH_OK();
    return AVD_OK;
}

}  // namespace wgrad3
}  // namespace avd
