// avd_env.cu -- batched vehicle-platoon environment for sm_100a.
//
// One thread owns one platoon and walks its followers in index order, exactly like Platoon.step's
// loop (/root/reference/src/environment.py:224-232), so the follower-order semantics (Model B
// exogenous input = predecessor's action of this step, Model A = predecessor's post-update
// acceleration, reset chaining of a_lead) need no inter-thread communication.  All arrays are
// struct-of-arrays with the platoon index fastest, so every load/store of a warp is one fully
// coalesced 128-byte line; a thread issues 6..9 independent loads per follower before its first
// dependent use (memory-level parallelism for an HBM-bound kernel: ~60 flop vs >=48 B per vehicle-step).
//
// Fused into the step when the corresponding pointers are given: OU exploration noise + action clip
// (src/noise.py:14-23, agent/ddpgagent.py:18-29), the leader's exogenous draw (workers/trainer.py:
// 292-295), ReplayBuffer.add for every agent (src/replaybuffer.py:37-47), episodic reward accumulation
// (workers/trainer.py:321), per-step reward/done statistics (block reduction + one atomic per CTA) and
// per-platoon auto-reset (src/environment.py:284-301, 520-559).
#include <cstdlib>

#include "avd_common.cuh"
#include "avd_rng.cuh"

namespace avd {

// ------------------------------------------------------------------------------------------------
// end of an episode for one platoon: publish the episodic reward counters (trainer.py:510-517: all_ep_reward_lists.append) and
// zero them (trainer.py:249).  `ep` = value of episode[p] before this reset = resets so far, so the finished episode is ep - 1.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void finish_episode(const avd_env_io& io, float* ep_reward, int M, int64_t p, uint32_t ep, bool stepped) {
    if (!ep_reward) return;
    const int64_t P = io.P;
    const int64_t hslot = (io.ep_hist && io.ep_hist_window > 0) ? (int64_t)((ep ? ep - 1u : 0u) % (uint32_t)io.ep_hist_window) : 0;
    for (int m = 0; m < M; ++m) {
        const int64_t v = (int64_t)m * P + p;
        if (stepped) {
            const float r = ep_reward[v];
            if (io.last_ep_reward) io.last_ep_reward[v] = r;
            if (io.ep_hist && io.ep_hist_window > 0) io.ep_hist[(hslot * M + m) * P + p] = r;
        }
        ep_reward[v] = 0.0f;
    }
}

// ------------------------------------------------------------------------------------------------
// reset of one platoon (thread-local): Platoon.reset + Vehicle.reset
// ------------------------------------------------------------------------------------------------
// `runs`: the run table (a kernel parameter), or a null constant in the instantiations that serve one run (they then compile to the
// code without run tables).
__device__ __forceinline__ void reset_one_platoon(const avd_env_params& prm, const avd_env_io& io, const avd_runs* runs, int64_t p,
                                                  uint32_t ep_tick, float* __restrict__ x_dst) {
    const int M = prm.M;
    const int64_t P = io.P;
    const StreamKey key = platoon_key(runs, io.seed, (uint64_t)(io.platoon_id_base + p));
    const uint64_t gp = key.id;
    const bool uni = prm.rand_uniform != 0;
    const uint4 wp = rng_words(key.seed, gp, ep_tick, AVD_RNG_RESET_PLATOON);
    float fa, fu;
    if (uni) {
        fa = uniform_sym(wp.x, prm.reset_leader_a);
        fu = uniform_sym(wp.y, prm.reset_u);
    } else {
        float z0, z1;
        normal_pair(wp.x, wp.y, z0, z1);
        fa = __fmul_rn(z0, prm.reset_leader_a);
        fu = __fmul_rn(z1, prm.reset_u);
    }
    if (io.front_accel) io.front_accel[p] = fa;
    if (io.front_u) io.front_u[p] = fu;
    float a_lead = fa;
    for (int m = 0; m < M; ++m) {
        float e0, e1, a;
        if (prm.reset_mode == 0) {
            const uint4 wv = rng_words(key.seed, gp * (uint64_t)M + (uint64_t)m, ep_tick, AVD_RNG_RESET_VEHICLE);
            if (uni) {
                e0 = uniform_sym(wv.x, prm.reset_ep);
                e1 = uniform_sym(wv.y, prm.reset_ev);
                a = uniform_sym(wv.z, prm.reset_a);
            } else {
                float z0, z1, z2, z3;
                normal_pair(wv.x, wv.y, z0, z1);
                normal_pair(wv.z, wv.w, z2, z3);
                e0 = __fmul_rn(z0, prm.reset_ep);
                e1 = __fmul_rn(z1, prm.reset_ev);
                a = __fmul_rn(z2, prm.reset_a);
            }
        } else {  // fixed maxima / evaluator states (environment.py:534-544, 551-555)
            e0 = prm.reset_ep;
            e1 = prm.reset_ev;
            a = prm.reset_a;
        }
        const int64_t v = (int64_t)m * P + p;
        x_dst[(0 * (int64_t)M) * P + v] = e0;
        x_dst[(1 * (int64_t)M) * P + v] = e1;
        x_dst[(2 * (int64_t)M) * P + v] = a;
        x_dst[(3 * (int64_t)M) * P + v] = a_lead;  // leader accel (m=0) or predecessor's fresh x[2]
        io.prev_a[v] = a;                          // prev_x = x (environment.py:557)
        if (io.cum_accel) io.cum_accel[v] = 0.0f;
        a_lead = a;
    }
    if (io.step_in_episode) io.step_in_episode[p] = 0;
}

template <bool RUNS>
__global__ void __launch_bounds__(256) env_reset_kernel(const __grid_constant__ avd_env_params prm,
                                                        const __grid_constant__ avd_env_io io,
                                                        const uint8_t* __restrict__ mask, const __grid_constant__ avd_runs rt) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < io.P; p += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[p]) continue;
        const uint32_t ep = io.episode ? (uint32_t)io.episode[p] : 0u;
        finish_episode(io, io.ep_reward, prm.M, p, ep, io.step_in_episode ? io.step_in_episode[p] > 0 : false);
        reset_one_platoon(prm, io, RUNS ? &rt : nullptr, p, ep, io.x_out);
        if (io.episode) io.episode[p] = (int32_t)(ep + 1u);
    }
}

// ------------------------------------------------------------------------------------------------
// step
// ------------------------------------------------------------------------------------------------
// Everything one follower needs from HBM; loaded for ALL followers of a platoon before the first dependent
// use so that a thread has 6..8 x M independent requests in flight (the kernel is HBM-latency/bandwidth bound).
struct FollowerIn {
    float x0, x1, x2, x3, pa, mu, ou, cum;
};

struct StepCtx {
    const float* __restrict__ x_in;
    float* __restrict__ x_out;
    float* __restrict__ prev_a;
    const float* __restrict__ action_mu;
    float* __restrict__ ou_state;
    float* __restrict__ action_out;
    float* __restrict__ reward;
    float* __restrict__ cum_accel;
    float* __restrict__ ep_reward;
    float* __restrict__ ring;
    float* __restrict__ jerk;
    float* __restrict__ velocity;
    float* __restrict__ headway;
    int64_t P, plane, slot;
    uint32_t tick;
    float inv_max_ep, inv_max_ev, inv_ahigh, inv_2maxa, inv_T, ou_c;
};

__device__ __forceinline__ FollowerIn load_follower(const StepCtx& c, int64_t v) {
    FollowerIn f;
    f.x0 = c.x_in[v];
    f.x1 = c.x_in[c.plane + v];
    f.x2 = c.x_in[2 * c.plane + v];
    f.x3 = c.x_in[3 * c.plane + v];
    f.pa = c.prev_a[v];
    f.mu = c.action_mu[v];
    f.ou = c.ou_state ? c.ou_state[v] : 0.0f;
    f.cum = c.cum_accel ? c.cum_accel[v] : 0.0f;
    return f;
}

// One Vehicle.step (environment.py:460-518) + fused OU/clip/replay write.  `w` is this follower's exogenous
// input on entry and the next follower's on exit.  Returns the (negated) reward; sets `term`.
// (Sharing one Philox block + Box-Muller transform between two followers -- z0 / z1 -- was measured in round 2: 5 % slower at M = 4,
// 3 % faster at M = 8, 10 % slower plain M = 8 launches from the changed register allocation; every follower keeps its own block.)
// ou_theta / ou_c: the platoon's OU theta and sigma * sqrt(dt) (its run's values when the batch holds several runs).
__device__ __forceinline__ float step_follower(const avd_env_params& prm, const avd_env_io& io, const StepCtx& c,
                                               const FollowerIn& f, int m, int M, int64_t p, StreamKey key, float ou_theta, float ou_c,
                                               float& w, bool& term) {
    const int64_t v = (int64_t)m * c.P + p;
    float u = f.mu;
    if (c.ou_state) {  // noise.py:14-23 with explicit single roundings (bit-exact vs the host restatement)
        float z0, z1;
        const uint4 wo = rng_words(key.seed, key.id * (uint64_t)M + (uint64_t)m, c.tick, AVD_RNG_OU);
        normal_pair(wo.x, wo.y, z0, z1);
        const float drift = __fmul_rn(__fmul_rn(ou_theta, __fadd_rn(prm.ou_mean, -f.ou)), prm.ou_dt);
        const float n1 = __fadd_rn(__fadd_rn(f.ou, drift), __fmul_rn(ou_c, z0));
        c.ou_state[v] = n1;
        u = __fadd_rn(u, n1);
    }
    if (io.clip_actions) u = fminf(fmaxf(u, prm.action_low), prm.action_high);  // ddpgagent.py:27
    if (c.action_out) c.action_out[v] = u;

    // reward terms on the PRE-update state (environment.py:473-477, 505-510)
    const float da = f.x2 - f.pa;
    const float r_shaped = (prm.rew_ep * (fabsf(f.x0) * c.inv_max_ep) + prm.rew_ev * (fabsf(f.x1) * c.inv_max_ev) +
                            prm.rew_u * (fabsf(u) * c.inv_ahigh) + prm.rew_jerk * (fabsf(da) * c.inv_2maxa)) * prm.re_scalar;
    term = prm.can_terminate && (fabsf(f.x0) > prm.max_ep || fabsf(f.x1) > prm.max_ev);
    const float r = -(term ? prm.terminal_reward * prm.re_scalar : r_shaped);  // Vehicle.step returns -reward
    if (c.jerk) c.jerk[v] = da * c.inv_T;
    if (c.cum_accel) {  // environment.py:500-503
        const float cum = f.cum + f.x2;
        c.cum_accel[v] = cum;
        const float vel = cum * prm.T;
        if (c.velocity) c.velocity[v] = vel;
        if (c.headway) c.headway[v] = f.x0 + (8.0f + prm.h * vel);
    }
    // x <- A x + B u + C w  (environment.py:513)
    const float* A = prm.A[m];
    const float* B = prm.B[m];
    const float* C = prm.C[m];
    const float y0 = fmaf(A[0], f.x0, fmaf(A[1], f.x1, fmaf(A[2], f.x2, fmaf(A[3], f.x3, fmaf(B[0], u, C[0] * w)))));
    const float y1 = fmaf(A[4], f.x0, fmaf(A[5], f.x1, fmaf(A[6], f.x2, fmaf(A[7], f.x3, fmaf(B[1], u, C[1] * w)))));
    const float y2 = fmaf(A[8], f.x0, fmaf(A[9], f.x1, fmaf(A[10], f.x2, fmaf(A[11], f.x3, fmaf(B[2], u, C[2] * w)))));
    const float y3 = fmaf(A[12], f.x0, fmaf(A[13], f.x1, fmaf(A[14], f.x2, fmaf(A[15], f.x3, fmaf(B[3], u, C[3] * w)))));
    c.x_out[v] = y0;
    c.x_out[c.plane + v] = y1;
    c.x_out[2 * c.plane + v] = y2;
    c.x_out[3 * c.plane + v] = y3;
    c.prev_a[v] = f.x2;
    if (!prm.centralized) c.reward[v] = r;
    if (c.ep_reward) c.ep_reward[v] += r;
    if (c.ring) {  // ReplayBuffer.add: (s, a, r, s') -- one 40 B record, five 8-byte stores.  (A warp's 32 records are contiguous, 1280 B;
                   // staging them through shared memory and writing 16-byte lines was measured in round 2 and dropped: +3..6 % launch
                   // time -- the launch is bound by the 30 / 70 read / write mix at the DRAM, not by the store instructions.)
        float2* rec = reinterpret_cast<float2*>(c.ring + ((c.slot * M + m) * c.P + p) * AVD_RING_RECORD_FLOATS);
        rec[0] = make_float2(f.x0, f.x1);
        rec[1] = make_float2(f.x2, f.x3);
        rec[2] = make_float2(u, r);
        rec[3] = make_float2(y0, y1);
        rec[4] = make_float2(y2, y3);
    }
    w = prm.model_a ? y2 : u;  // next follower's exogenous input (environment.py:261 / 267)
    return r;
}

// Registers: the preloaded inputs cost 8 per follower.  Platoons of up to 4 followers are preloaded whole; longer ones in chunks of 4
// (the exogenous input `w` carries the chain from chunk to chunk), so every instantiation fits 80 registers = 3 CTAs per SM --
// preloading all 8 followers needed 128 registers (2 CTAs per SM) and left the M = 8 launches 15 % behind the M = 4 ones.
// TRAIN (OU noise / replay ring fused: the launch of the training loop) is compute-heavier per vehicle (Philox + Box-Muller per
// follower) than the plain step, so it trades loads in flight per thread for more resident warps: 4 CTAs per SM (64 registers), and
// for platoons longer than 4 chunks of 2 followers, which fit 64 registers without spilling.  Measured on 4 Mi platoons (launch
// time, us; `chunk / CTAs per SM`):      M = 4:  4/3 428   4/4 370   2/4 388   2/5 388        M = 8:  4/3 881   4/4 1002   2/4 829   2/5 959
// RUNS: the batch holds several runs (rt, a copy of *io.runs); a separate instantiation because the run-table lookup costs registers.
// Only these instantiations read the optional per-run OU parameters (rt.ou_sigma / rt.ou_theta).
template <int MT, bool TRAIN, bool RUNS>
__global__ void __launch_bounds__(256, MT >= 1 ? (TRAIN ? 4 : 3) : 2)
    env_step_kernel(const __grid_constant__ avd_env_params prm, const __grid_constant__ avd_env_io io, const __grid_constant__ avd_runs rt) {
    const int M = MT ? MT : prm.M;
    StepCtx c;
    c.x_in = io.x_in; c.x_out = io.x_out; c.prev_a = io.prev_a; c.action_mu = io.action_mu; c.ou_state = io.ou_state;
    c.action_out = io.action_out; c.reward = io.reward; c.cum_accel = io.cum_accel; c.ep_reward = io.ep_reward;
    c.ring = io.ring; c.jerk = io.jerk; c.velocity = io.velocity; c.headway = io.headway;
    c.P = io.P;
    c.plane = (int64_t)M * io.P;  // one state component of all vehicles
    const uint64_t tick64 = io.clock ? io.clock->step_tick : 0ull;
    c.tick = (uint32_t)tick64;
    const uint64_t ring_count = io.clock ? io.clock->ring_count : 0ull;
    c.slot = io.ring ? (int64_t)(ring_count % (uint64_t)io.ring_capacity) : 0;
    const bool uni = prm.rand_uniform != 0;
    c.inv_max_ep = 1.0f / prm.max_ep; c.inv_max_ev = 1.0f / prm.max_ev;
    c.inv_ahigh = 1.0f / fabsf(prm.action_high); c.inv_2maxa = 1.0f / (2.0f * prm.action_high);
    c.inv_T = 1.0f / prm.T;
    c.ou_c = __fmul_rn(prm.ou_sigma, __fsqrt_rn(prm.ou_dt));
    const int64_t P = io.P;
    const avd_runs* runs = RUNS ? &rt : nullptr;

    float stat_r[MT ? MT : AVD_MAX_FOLLOWERS];
#pragma unroll
    for (int m = 0; m < (MT ? MT : AVD_MAX_FOLLOWERS); ++m) stat_r[m] = 0.0f;
    float stat_done = 0.0f;

    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (int64_t)gridDim.x * blockDim.x) {
        const StreamKey key = platoon_key(runs, io.seed, (uint64_t)(io.platoon_id_base + p));
        float ou_theta = prm.ou_theta, ou_c = c.ou_c;
        if (RUNS && TRAIN) {      // (a plain step has no OU noise)
            const uint64_t run = (uint64_t)p / (uint64_t)rt.platoons_per_run;
            if (rt.ou_theta) ou_theta = rt.ou_theta[run];
            if (rt.ou_sigma) ou_c = __fmul_rn(rt.ou_sigma[run], __fsqrt_rn(prm.ou_dt));
        }
        constexpr int CH = MT > 4 ? (TRAIN ? 2 : 4) : (MT ? MT : 1);       // followers preloaded at a time
        FollowerIn fin[CH];
        if (MT) {
#pragma unroll
            for (int m = 0; m < CH; ++m) fin[m] = load_follower(c, (int64_t)m * P + p);
        }
        // exogenous input of follower 0 (environment.py:258-259 / 264-265, trainer.py:292-295)
        float w;
        if (io.leader_exog) {
            w = io.leader_exog[p];
        } else if (io.gen_exog) {
            const uint4 wx = rng_words(key.seed, key.id, c.tick, AVD_RNG_LEADER_EXOG);
            w = draw_first(wx.x, wx.y, prm.reset_u, uni);
        } else {
            w = prm.model_a ? io.front_accel[p] : io.front_u[p];
        }
        bool any_term = false;
        float rew_sum = 0.0f;
        if (MT) {
#pragma unroll
            for (int m0 = 0; m0 < MT; m0 += CH) {
                if (m0 > 0) {
#pragma unroll
                    for (int j = 0; j < CH; ++j)
                        if (m0 + j < MT) fin[j] = load_follower(c, (int64_t)(m0 + j) * P + p);
                }
#pragma unroll
                for (int j = 0; j < CH; ++j) {
                    if (m0 + j < MT) {
                        bool term;
                        const float r = step_follower(prm, io, c, fin[j], m0 + j, MT, p, key, ou_theta, ou_c, w, term);
                        any_term |= term;
                        rew_sum += r;
                        stat_r[m0 + j] += r;
                    }
                }
            }
        } else {
            for (int m = 0; m < M; ++m) {
                bool term;
                const FollowerIn f = load_follower(c, (int64_t)m * P + p);
                const float r = step_follower(prm, io, c, f, m, M, p, key, ou_theta, ou_c, w, term);
                any_term |= term;
                rew_sum += r;
                stat_r[m] += r;
            }
        }
        if (prm.centralized) io.reward[p] = rew_sum * (1.0f / (float)M);  // environment.py:281
        bool timeout = false;
        if (io.step_in_episode) {
            const int s = io.step_in_episode[p] + 1;
            timeout = prm.steps_per_episode > 0 && s >= prm.steps_per_episode;
            io.step_in_episode[p] = s;
        }
        io.done[p] = (uint8_t)((any_term ? 1 : 0) | (timeout ? 2 : 0));
        stat_done += any_term ? 1.0f : 0.0f;
        if (io.auto_reset && (any_term || timeout)) {
            const uint32_t ep = io.episode ? (uint32_t)io.episode[p] : 0u;
            finish_episode(io, c.ep_reward, M, p, ep, true);
            reset_one_platoon(prm, io, runs, p, ep, io.x_out);
            if (io.episode) io.episode[p] = (int32_t)(ep + 1u);
        }
    }

    if (io.stats) {  // warp shuffle -> shared -> one atomic per CTA and statistic
        __shared__ float red[8][AVD_MAX_FOLLOWERS + 1];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
        for (int m = 0; m < (MT ? MT : AVD_MAX_FOLLOWERS); ++m) {
            const float s = warp_sum(stat_r[m]);
            if (lane == 0) red[wid][m] = s;
        }
        const float sd = warp_sum(stat_done);
        if (lane == 0) red[wid][AVD_MAX_FOLLOWERS] = sd;
        __syncthreads();
        if (threadIdx.x <= M) {
            const int col = (threadIdx.x == M) ? AVD_MAX_FOLLOWERS : threadIdx.x;
            float s = 0.0f;
            for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) s += red[wv][col];
            atomicAdd(io.stats + threadIdx.x, s);
        }
    }
}

__global__ void __launch_bounds__(256) ou_sample_kernel(float theta, float mean, float dt, float sigma, float* __restrict__ state,
                                                        float* __restrict__ out, int64_t n, uint64_t id_base, uint64_t seed,
                                                        uint32_t tick) {
    const float ou_c = __fmul_rn(sigma, __fsqrt_rn(dt));
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float n0 = state[i];
        const uint4 wo = rng_words(seed, id_base + (uint64_t)i, tick, AVD_RNG_OU);
        float z0, z1;
        normal_pair(wo.x, wo.y, z0, z1);
        const float drift = __fmul_rn(__fmul_rn(theta, __fadd_rn(mean, -n0)), dt);
        const float n1 = __fadd_rn(__fadd_rn(n0, drift), __fmul_rn(ou_c, z0));
        state[i] = n1;
        if (out) out[i] = n1;
    }
}

__global__ void clock_advance_kernel(avd_clock* c, uint32_t ds, uint32_t dr, uint32_t du) {
    c->step_tick += ds;
    c->ring_count += dr;
    c->update_tick += du;
}

static int check_env_args(const avd_env_params* prm, const avd_env_io* io) {
    AVD_REQUIRE(prm && io, "null params");
    AVD_REQUIRE(prm->M >= 1 && prm->M <= AVD_MAX_FOLLOWERS, "M=%d outside 1..%d", prm->M, AVD_MAX_FOLLOWERS);
    AVD_REQUIRE(io->P >= 0, "negative platoon count");
    AVD_REQUIRE(io->P == 0 || io->prev_a, "prev_a buffer is required");
    if (io->runs) {
        AVD_REQUIRE(io->platoon_id_base == 0, "a run table indexes the whole batch: platoon_id_base must be 0");
        AVD_REQUIRE_RUNS(io->runs, io->P);
    }
    return AVD_OK;
}

}  // namespace avd

using namespace avd;

extern "C" int avd_clock_advance(avd_clock* clock_dev, uint32_t d_step, uint32_t d_ring, uint32_t d_update, void* stream) {
    AVD_REQUIRE(clock_dev, "null clock");
    clock_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(clock_dev, d_step, d_ring, d_update);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_ou_sample(const avd_env_params* prm, float* state, float* out, int64_t n, uint64_t id_base, uint64_t seed,
                             uint32_t tick, void* stream) {
    AVD_REQUIRE(prm && state && n >= 0, "bad args");
    if (n == 0) return AVD_OK;
    ou_sample_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(prm->ou_theta, prm->ou_mean, prm->ou_dt, prm->ou_sigma, state, out,
                                                                     n, id_base, seed, tick);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_env_reset(const avd_env_params* prm, const avd_env_io* io, const uint8_t* mask, void* stream) {
    if (int rc = check_env_args(prm, io)) return rc;
    if (io->P == 0) return AVD_OK;
    AVD_REQUIRE(io->x_out, "x_out is required");
    if (io->runs) env_reset_kernel<true><<<grid_for(io->P), 256, 0, (cudaStream_t)stream>>>(*prm, *io, mask, *io->runs);
    else env_reset_kernel<false><<<grid_for(io->P), 256, 0, (cudaStream_t)stream>>>(*prm, *io, mask, avd_runs{});
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_env_step(const avd_env_params* prm, const avd_env_io* io, void* stream) {
    if (int rc = check_env_args(prm, io)) return rc;
    if (io->P == 0) return AVD_OK;
    AVD_REQUIRE(io->x_in && io->x_out && io->action_mu && io->reward && io->done, "x_in/x_out/action_mu/reward/done are required");
    AVD_REQUIRE(io->x_in != io->x_out, "x_in and x_out must not alias (ping-pong state buffers)");
    AVD_REQUIRE(!io->ring || io->ring_capacity > 0, "ring given with capacity %lld", (long long)io->ring_capacity);
    AVD_REQUIRE(!io->auto_reset || (io->episode && io->step_in_episode), "auto_reset needs episode and step_in_episode");
    AVD_REQUIRE(!io->ep_hist || (io->ep_hist_window > 0 && io->ep_reward && io->episode), "ep_hist needs a window, ep_reward and episode counters");
    AVD_REQUIRE(io->leader_exog || io->gen_exog || (prm->model_a ? io->front_accel != nullptr : io->front_u != nullptr),
                "no source for the leader's exogenous input");
    if (io->P == 0) return AVD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const bool train = io->ring != nullptr || io->ou_state != nullptr;
    const avd_runs rt = io->runs ? *io->runs : avd_runs{};
#define AVD_LAUNCH_STEP_R(MT, RUNS)                                                                                                    \
    do {                                                                                                                               \
        if (train) env_step_kernel<MT, true, RUNS><<<resident_grid(env_step_kernel<MT, true, RUNS>, io->P), 256, 0, st>>>(*prm, *io, rt); \
        else env_step_kernel<MT, false, RUNS><<<resident_grid(env_step_kernel<MT, false, RUNS>, io->P), 256, 0, st>>>(*prm, *io, rt);   \
    } while (0)
#define AVD_LAUNCH_STEP(MT)                          \
    do {                                             \
        if (io->runs) AVD_LAUNCH_STEP_R(MT, true);   \
        else AVD_LAUNCH_STEP_R(MT, false);           \
    } while (0)
    switch (prm->M) {
        case 1: AVD_LAUNCH_STEP(1); break;
        case 2: AVD_LAUNCH_STEP(2); break;
        case 3: AVD_LAUNCH_STEP(3); break;
        case 4: AVD_LAUNCH_STEP(4); break;
        case 5: AVD_LAUNCH_STEP(5); break;
        case 6: AVD_LAUNCH_STEP(6); break;
        case 8: AVD_LAUNCH_STEP(8); break;
        default: AVD_LAUNCH_STEP(0); break;
    }
#undef AVD_LAUNCH_STEP
#undef AVD_LAUNCH_STEP_R
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_env_step_host(const avd_env_params* prm, const avd_env_io* io, const float* actions_host,
                                 const float* leader_exog_host, float* obs_host, float* reward_host,
                                 uint8_t* done_host, void* stream) {
    if (int rc = check_env_args(prm, io)) return rc;
    if (io->P == 0) return AVD_OK;
    AVD_REQUIRE(actions_host && obs_host && reward_host && done_host, "null host buffer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)prm->M * (size_t)io->P;
    AVD_CUDA_OK(cudaMemcpyAsync((void*)io->action_mu, actions_host, n * sizeof(float), cudaMemcpyHostToDevice, st));
    if (leader_exog_host) {
        AVD_REQUIRE(io->leader_exog, "leader_exog_host given but io->leader_exog staging is NULL");
        AVD_CUDA_OK(cudaMemcpyAsync((void*)io->leader_exog, leader_exog_host, (size_t)io->P * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    if (int rc = avd_env_step(prm, io, stream)) return rc;
    AVD_CUDA_OK(cudaMemcpyAsync(obs_host, io->x_out, 4 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
    AVD_CUDA_OK(cudaMemcpyAsync(reward_host, io->reward, (prm->centralized ? (size_t)io->P : n) * sizeof(float), cudaMemcpyDeviceToHost, st));
    AVD_CUDA_OK(cudaMemcpyAsync(done_host, io->done, (size_t)io->P, cudaMemcpyDeviceToHost, st));
    AVD_CUDA_OK(cudaStreamSynchronize(st));
    return AVD_OK;
}

extern "C" int avd_env_build_matrices(avd_env_params* prm, int method, double T, double h, double tau,
                                      double pl_leader_tau) {
    AVD_REQUIRE(prm, "null params");
    AVD_REQUIRE(prm->M >= 1 && prm->M <= AVD_MAX_FOLLOWERS, "M=%d outside 1..%d", prm->M, AVD_MAX_FOLLOWERS);
    AVD_REQUIRE(method == 0 || method == 1, "method must be 0 (euler) or 1 (exact)");
    AVD_REQUIRE(T > 0 && tau > 0 && pl_leader_tau > 0, "sample_rate, dyn_coeff and pl_leader_tau must be positive");
    prm->T = (float)T;
    prm->h = (float)h;
    for (int m = 0; m < prm->M; ++m) {
        const double tl = (m == 0) ? pl_leader_tau : tau;
        double A[16] = {0}, B[4] = {0}, C[4] = {0};
        A[0] = 1.0; A[1] = T; A[5] = 1.0;
        if (method == 0) {  // environment.py:393-408
            A[2] = -h * T;
            A[6] = -T; A[7] = T;
            A[10] = 1.0 - T / tau;
            A[15] = 1.0 - T / tl;
            B[2] = T / tau;
            C[3] = T / tl;
        } else {            // environment.py:410-445
            const double e = exp(-T / tau), el = exp(-T / tl);
            A[2] = -h * tau + h * tau * e - tau * T + tau * tau - tau * tau * e;
            A[3] = tl * T - tl * tl + tl * tl * el;
            A[6] = -tau + tau * e;
            A[7] = tl - tl * el;
            A[10] = e;
            A[15] = el;
            B[0] = -h * T + h * tau * e - h * tau - T * T / 2 + tau * T + tau * tau * e - tau * tau;
            B[1] = -T - tau * e + tau;
            B[2] = 1.0 - e;
            C[0] = T * T / 2 - tl * T - tl * tl * el + tl * tl;
            C[1] = T + tl * el - tl;
            C[3] = 1.0 - el;
        }
        for (int i = 0; i < 16; ++i) prm->A[m][i] = (float)A[i];
        for (int i = 0; i < 4; ++i) { prm->B[m][i] = (float)B[i]; prm->C[m][i] = (float)C[i]; }
    }
    return AVD_OK;
}
