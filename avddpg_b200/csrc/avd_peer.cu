// avd_peer.cu -- the exchange step of the federated (interfrl) round as NVLink-native kernels.
//
//   every rank has written its per-system partial sums [systems][pitch] (last used column = the local member count or
//   weight sum) into its half of a SYMMETRIC buffer (same offset in every rank's peer-mapped allocation); the kernels here
//     1. signal "my partial sums are complete" into every peer's flag word and wait for all peers' signals
//        (st.release.sys / ld.acquire.sys on peer-mapped memory, monotonically increasing epoch, no reset),
//     2. read the SUM over ranks -- with `multimem.ld_reduce` on the NVLS multicast mapping, i.e. reduced inside the
//        NVSwitch, or, without a multicast mapping, with plain peer loads over NVLink --
//     3. divide by the reduced count / weight sum (federated.py:62, :110) and
//          fed_exchange_peer_kernel : write the means to local memory (weights mode: set_weights follows, trainer.py:448-456)
//          fed_apply_kernel         : CONSUME them on the spot -- every local member of the system takes its tf.keras Adam step
//                                     with the averaged gradient and soft-updates its target network (trainer.py:419-431), so a
//                                     gradients round is  fed_reduce2 -> this kernel  and the averaged gradients never travel
//                                     through HBM again (round 1: reduce -> exchange -> broadcast -> Adam/Polyak -> step counters).
// The epoch lives in DEVICE memory (ctrl[0], advanced by the last CTA of each exchange kernel), so a CUDA graph that contains a
// round replays correctly: nothing about the barrier is baked into the launch arguments.
// Buffers alternate between two halves from round to round: a rank can only pass the barrier of round k+1 after every
// peer has finished reading round k, so half (k & 1) is free again when round k+2 writes it.
#include "avd_common.cuh"

namespace avd {

struct PeerCore {
    int rank, world;
    uint64_t peer_base[AVD_MAX_PEERS];     // peer-mapped base address of every rank's symmetric allocation
    uint64_t multicast_base;               // NVLS multicast mapping of the same allocation (0: none)
    int64_t flag_off, data_off;            // byte offsets inside the allocation: epoch flags [AVD_MAX_PEERS] u32, partial sums
    const float* local;                    // world == 1: the partial sums in plain local memory (no exchange)
    uint32_t* ctrl;                        // local device memory: [0] rounds completed (epoch), [1] CTAs finished in this round,
                                           // [2] 0, or 1 + the first peer rank whose signal did not arrive within the time limit
    long long timeout_cycles;              // spin limit of the barrier (SM clock cycles)
    int64_t pitch;                         // floats per system row (multiple of 4)
    int n_systems;
    int64_t n;                             // payload columns; column n carries the divisor
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 multimem_sum4(const float* mc) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
    return v;
}

// cross-rank barrier of this round: block 0 signals, every block waits on the LOCAL flag words
__device__ __forceinline__ void peer_barrier(const PeerCore& g) {
    if (g.world > 1) {
        const uint32_t epoch = *reinterpret_cast<volatile uint32_t*>(g.ctrl) + 1u;     // only the last CTA of a round advances it
        if (blockIdx.x == 0 && threadIdx.x < g.world) {
            __threadfence_system();
            st_release_sys(reinterpret_cast<uint32_t*>(g.peer_base[threadIdx.x] + g.flag_off) + g.rank, epoch);
        }
        if (threadIdx.x < g.world) {
            const uint32_t* flag = reinterpret_cast<const uint32_t*>(g.peer_base[g.rank] + g.flag_off) + threadIdx.x;
            // A peer that never issues this round (a rank that fell back to another transport, died, or runs a different schedule)
            // must not hang the GPU for good: after the time limit the wait gives up, records the missing rank in ctrl[2] and the
            // round completes with whatever the buffers hold -- avd_fed_round_status / PeerExchange.check() turn that into an error.
            const long long t0 = clock64();
            while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
                if (clock64() - t0 > g.timeout_cycles) {
                    atomicCAS(g.ctrl + 2, 0u, 1u + threadIdx.x);
                    break;
                }
            }
        }
    }
    __syncthreads();
}

// float4 chunk at byte offset `off` of the symmetric data region, summed over the ranks
__device__ __forceinline__ float4 peer_sum4(const PeerCore& g, int64_t off) {
    if (g.world <= 1) return *reinterpret_cast<const float4*>(reinterpret_cast<const char*>(g.local) + off);
    if (g.multicast_base) return multimem_sum4(reinterpret_cast<const float*>(g.multicast_base + g.data_off + off));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = 0; r < g.world; ++r) {
        const float4 a = *reinterpret_cast<const float4*>(g.peer_base[r] + g.data_off + off);
        v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    return v;
}

// 1 / (reduced divisor of system s); also hands the divisor itself back
__device__ __forceinline__ float peer_inv_divisor(const PeerCore& g, int s, float& divisor) {
    const float4 dv = peer_sum4(g, ((int64_t)s * g.pitch + (g.n & ~(int64_t)3)) * 4);      // float4 that holds the divisor column
    const int k = (int)(g.n & 3);
    divisor = k == 0 ? dv.x : k == 1 ? dv.y : k == 2 ? dv.z : dv.w;
    return 1.0f / divisor;
}

// last CTA of the round: returns true for exactly one CTA, after ALL CTAs of this launch have called it
__device__ __forceinline__ bool peer_round_done(const PeerCore& g) {
    __shared__ int last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(g.ctrl + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        g.ctrl[1] = 0u;
        __threadfence();
        *reinterpret_cast<volatile uint32_t*>(g.ctrl) = g.ctrl[0] + 1u;
    }
    return last != 0;
}

__global__ void __launch_bounds__(256) fed_exchange_peer_kernel(PeerCore g, float* __restrict__ out) {
    peer_barrier(g);
    const int64_t row_f4 = g.pitch / 4;
    const int64_t total = (int64_t)g.n_systems * row_f4;
    int cur_s = -1;
    float inv = 0.0f, divisor = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int s = (int)(i / row_f4);
        const int64_t c4 = (i - (int64_t)s * row_f4) * 4;
        if (s != cur_s) { inv = peer_inv_divisor(g, s, divisor); cur_s = s; }      // once per row and thread, not per chunk
        const float4 v = peer_sum4(g, ((int64_t)s * g.pitch + c4) * 4);
        float* dst = out + (int64_t)s * g.pitch + c4;
        const float raw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)      // payload columns: the mean; column n: the reduced divisor itself (fed_weight_sums, trainer.py:358-359)
            if (c4 + j <= g.n) dst[j] = c4 + j < g.n ? raw[j] * inv : raw[j];
    }
    peer_round_done(g);
}

// ---- fused consumer -----------------------------------------------------------------------------------
struct ApplyNet {
    float *params, *target, *m, *v;        // [A][total] / [A][n_train]
    int32_t* step;                         // [A] Adam step counters (incremented by the last CTA)
    float* grad_out;                       // nullable: [A][n_train] the averaged gradient, written to every member (API parity)
    int64_t total, n_train;
    float lr;
};
struct ApplyArgs {
    PeerCore core;
    ApplyNet net[2];                       // columns [0, na) -> net[0] (actor), [na, na + nc) -> net[1] (critic)
    int n_members, A;
    int64_t stride_s, stride_x;            // member (s, x) = agent s*stride_s + x*stride_x
    const uint8_t* mask;                   // [A] nullable: agents with 0 keep their weights
    float b1, b2, eps, tau;
    float* wsum_out;                       // [systems] nullable: the reduced divisor
    const float* hp;                       // [A][4] (gamma, actor_lr, critic_lr, tau) per agent; read by the HP instantiation only
};

// HP: every agent takes its learning rates and tau from a.hp (same arithmetic as with the scalars); the table then holds [3][A]
// floats -- the two lr_t rows and tau -- instead of [2][A], which lowers the largest A from 25,600 to 17,066 (200 KB).
template <bool HP>
__global__ void __launch_bounds__(256) fed_apply_kernel(ApplyArgs a) {
    extern __shared__ float lr_tab[];      // [2][A]: lr * sqrt(1 - b2^t) / (1 - b1^t) per net and agent, t = step + 1;  HP: + [A] tau
    const PeerCore& g = a.core;
    for (int i = threadIdx.x; i < 2 * a.A; i += blockDim.x) {
        const ApplyNet& nt = a.net[i / a.A];
        const float t = (float)(nt.step[i % a.A] + 1);
        const float lr = HP ? a.hp[4 * (i % a.A) + (i < a.A ? 1 : 2)] : nt.lr;      // net[0] is the actor
        lr_tab[i] = lr * sqrtf(1.0f - powf(a.b2, t)) / (1.0f - powf(a.b1, t));
    }
    const float* tau_tab = lr_tab + 2 * a.A;
    if (HP)
        for (int i = threadIdx.x; i < a.A; i += blockDim.x) lr_tab[2 * a.A + i] = a.hp[4 * i + 3];
    peer_barrier(g);                       // ends with __syncthreads(): the table is complete
    const int64_t na = a.net[0].n_train;
    const float omt = 1.0f - a.tau;
    const int64_t row_f4 = g.pitch / 4;
    const int64_t total = (int64_t)g.n_systems * row_f4;
    int cur_s = -1;
    float inv = 0.0f, divisor = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int s = (int)(i / row_f4);
        const int64_t c4 = (i - (int64_t)s * row_f4) * 4;
        const float4 v4 = peer_sum4(g, ((int64_t)s * g.pitch + c4) * 4);      // issued before the divisor is needed: both loads in flight
        if (s != cur_s) { inv = peer_inv_divisor(g, s, divisor); cur_s = s; }
        const float raw[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t col = c4 + j;
            if (col > g.n) continue;
            if (col == g.n) {
                if (a.wsum_out) a.wsum_out[s] = raw[j];
                continue;
            }
            const int k = col < na ? 0 : 1;
            const ApplyNet& nt = a.net[k];
            const int64_t idx = k ? col - na : col;
            const float gavg = raw[j] * inv;                       // federated.py:62 / :110
            for (int x = 0; x < a.n_members; ++x) {
                const int64_t ag = (int64_t)s * a.stride_s + (int64_t)x * a.stride_x;
                if (a.mask && !a.mask[ag]) continue;
                if (nt.grad_out) nt.grad_out[ag * nt.n_train + idx] = gavg;
                // tf.keras Adam (trainer.py:420-425) then ddpgagent.update_target (428-431); same arithmetic as adam_polyak2_kernel
                float* Mm = nt.m + ag * nt.n_train + idx;
                float* Vv = nt.v + ag * nt.n_train + idx;
                float* Pp = nt.params + ag * nt.total + idx;
                float* Tt = nt.target + ag * nt.total + idx;
                const float mi = *Mm + (gavg - *Mm) * (1.0f - a.b1);
                const float vi = *Vv + (gavg * gavg - *Vv) * (1.0f - a.b2);
                *Mm = mi;
                *Vv = vi;
                const float p = *Pp - lr_tab[k * a.A + (int)ag] * mi / (sqrtf(vi) + a.eps);
                *Pp = p;
                if (HP) *Tt = p * tau_tab[ag] + *Tt * (1.0f - tau_tab[ag]);
                else *Tt = p * a.tau + *Tt * omt;
            }
        }
    }
    // the non-trainable tail (BatchNormalization moving statistics) only takes part in the soft update (ddpgagent.py:46-53)
    const int64_t tail0 = a.net[0].total - a.net[0].n_train, tail1 = a.net[1].total - a.net[1].n_train;
    const int64_t per_agent = tail0 + tail1, tails = per_agent * a.A;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < tails; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ag = i / per_agent, r = i - ag * per_agent;
        if (a.mask && !a.mask[ag]) continue;
        const ApplyNet& nt = a.net[r < tail0 ? 0 : 1];
        const int64_t idx = nt.n_train + (r < tail0 ? r : r - tail0);
        float* Tt = nt.target + ag * nt.total + idx;
        if (HP) *Tt = nt.params[ag * nt.total + idx] * tau_tab[ag] + *Tt * (1.0f - tau_tab[ag]);
        else *Tt = nt.params[ag * nt.total + idx] * a.tau + *Tt * omt;
    }
    if (peer_round_done(g)) {              // every CTA has built its lr table: the step counters may advance now
        for (int i = threadIdx.x; i < a.A; i += blockDim.x)
            if (!a.mask || a.mask[i]) { a.net[0].step[i] += 1; a.net[1].step[i] += 1; }
    }
}

static int fill_core(PeerCore& g, const avd_peer_comm* comm, int64_t flag_offset, int64_t data_offset, const float* local, uint32_t* ctrl,
                     int64_t pitch, int32_t n_systems, int64_t n) {
    AVD_REQUIRE(comm && ctrl, "null argument");
    AVD_REQUIRE(comm->world >= 1 && comm->world <= AVD_MAX_PEERS && comm->rank >= 0 && comm->rank < comm->world, "bad rank / world (max %d peers)", AVD_MAX_PEERS);
    AVD_REQUIRE(pitch % 4 == 0 && n >= 1 && n < pitch && n_systems >= 1, "pitch must be a multiple of 4 floats and hold n + 1 columns");
    AVD_REQUIRE(flag_offset % 4 == 0 && data_offset % 16 == 0, "misaligned offsets");
    AVD_REQUIRE(comm->world > 1 || (local && ((uintptr_t)local & 15) == 0), "a single rank needs its partial sums in 16-byte aligned local memory");
    g.rank = comm->rank; g.world = comm->world;
    for (int r = 0; r < AVD_MAX_PEERS; ++r) g.peer_base[r] = r < comm->world ? comm->peer_base[r] : 0;
    g.multicast_base = comm->world > 1 ? comm->multicast_base : 0;
    g.flag_off = flag_offset; g.data_off = data_offset; g.local = local; g.ctrl = ctrl; g.pitch = pitch; g.n_systems = n_systems; g.n = n;
    static const long long limit_ms = [] { const char* e = getenv("AVD_PEER_TIMEOUT_MS"); const long long v = e ? atoll(e) : 0; return v > 0 ? v : 20000ll; }();
    g.timeout_cycles = limit_ms * 2000000ll;      // ~2 GHz SM clock: the limit only has to be generous, not exact
    if (comm->world > 1)
        for (int r = 0; r < comm->world; ++r) AVD_REQUIRE(g.peer_base[r] != 0, "peer %d has no mapped buffer", r);
    return AVD_OK;
}

}  // namespace avd

extern "C" int avd_fed_exchange_peer(const avd_peer_comm* comm, int64_t flag_offset, int64_t data_offset, uint32_t* ctrl, float* out,
                                     int64_t pitch, int32_t n_systems, int64_t n, void* stream) {
    using namespace avd;
    AVD_REQUIRE(out, "null argument");
    PeerCore g;
    if (int rc = fill_core(g, comm, flag_offset, data_offset, out, ctrl, pitch, n_systems, n)) return rc;
    AVD_REQUIRE(comm->world > 1, "the peer exchange needs at least two ranks");
    const int64_t work = (int64_t)n_systems * (pitch / 4);
    // few CTAs: every one of them spins on the barrier flags, and 1-2.5 MB of payload needs no more than a few hundred loads in flight per SM
    const int grid = (int)std::min<int64_t>((work + 255) / 256, sm_count());
    fed_exchange_peer_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g, out);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_apply_gradients(const avd_fed_apply_io* io, void* stream) {
    using namespace avd;
    AVD_REQUIRE(io, "null io");
    ApplyArgs a = {};
    const int64_t n = io->actor_train + io->critic_train;
    if (int rc = fill_core(a.core, &io->comm, io->flag_offset, io->data_offset, io->local_sums, io->ctrl, io->pitch, io->n_systems, n)) return rc;
    AVD_REQUIRE(io->actor && io->t_actor && io->actor_m && io->actor_v && io->actor_step && io->critic && io->t_critic && io->critic_m && io->critic_v &&
                    io->critic_step,
                "null parameter / optimiser buffer");
    AVD_REQUIRE(io->A >= 1 && io->n_members >= 1 && io->actor_total >= io->actor_train && io->critic_total >= io->critic_train, "bad sizes");
    AVD_REQUIRE((int64_t)(io->n_systems - 1) * io->member_stride_s + (int64_t)(io->n_members - 1) * io->member_stride_x < io->A, "member indices exceed A");
    a.net[0] = ApplyNet{io->actor, io->t_actor, io->actor_m, io->actor_v, io->actor_step, io->actor_grad_out, io->actor_total, io->actor_train, io->actor_lr};
    a.net[1] = ApplyNet{io->critic, io->t_critic, io->critic_m, io->critic_v, io->critic_step, io->critic_grad_out, io->critic_total, io->critic_train, io->critic_lr};
    a.n_members = io->n_members; a.A = io->A; a.stride_s = io->member_stride_s; a.stride_x = io->member_stride_x; a.mask = io->apply_mask;
    a.b1 = io->beta1; a.b2 = io->beta2; a.eps = io->eps; a.tau = io->tau; a.wsum_out = io->wsum_out; a.hp = io->agent_hp;
    const bool hp = io->agent_hp != nullptr;
    const size_t smem = (size_t)(hp ? 3 : 2) * io->A * sizeof(float);
    AVD_REQUIRE(smem <= 200 * 1024, "too many agents per rank for the fused federated consumer (%d%s)", io->A, hp ? " with a per-agent table" : "");
    static size_t smem_set[2] = {48 * 1024, 0};      // with a table: set the limit on first use (the kernel also has static shared memory)
    if (smem > smem_set[hp]) {
        AVD_CUDA_OK(cudaFuncSetAttribute(hp ? fed_apply_kernel<true> : fed_apply_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set[hp] = smem;
    }
    const int64_t work = (int64_t)io->n_systems * (io->pitch / 4);
    const int grid = (int)std::min<int64_t>((work + 255) / 256, 2 * sm_count());
    if (hp) fed_apply_kernel<true><<<grid, 256, smem, (cudaStream_t)stream>>>(a);
    else fed_apply_kernel<false><<<grid, 256, smem, (cudaStream_t)stream>>>(a);
    AVD_LAUNCH_OK();
    return AVD_OK;
}
