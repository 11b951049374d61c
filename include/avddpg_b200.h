/* avddpg_b200.h -- C ABI of the B200-native avddpg hot path (libavddpg_b200.so).
 *
 * The reference (cboin1996/avddpg) is pure Python and has no FFI of its own; its boundary is the
 * Python call surface workers/trainer.py uses (SURVEY.md §8b).  Every entry point below names the
 * reference interface it replaces (file:line under /root/reference).  INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C: pointers, sizes, PODs.  No torch / C++ types cross this boundary.
 *   - every `*_dev` / unqualified buffer pointer is DEVICE memory of the current CUDA device;
 *     entry points whose name ends in `_host` take HOST pointers and do the copies themselves.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All calls are
 *     asynchronous with respect to the host unless the name ends in `_host` or `_sync`.
 *   - return value: 0 on success, negative avd_status on error; avd_last_error() gives the text.
 *     (The reference raises Python exceptions -- ValueError etc.; the Python mirror in
 *     avddpg_b200/ converts these codes back into the same exception types.)
 *   - layouts: platoon state is struct-of-arrays, platoon index fastest:
 *         x[f][m][p]  -> ((f*M + m)*P + p)      f in 0..3  (ep, ev, a, a_lead)
 *         per-vehicle scalars (action, reward, prev_a, ...)  [m][p] -> (m*P + p)
 *     replay ring records are array-of-structs, 10 floats each (s[4], a, r, s'[4]):
 *         ring[slot][m][p][10] -> (((slot*M + m)*P + p)*10)
 */
#ifndef AVDDPG_B200_H
#define AVDDPG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVD_MAX_FOLLOWERS 16
#define AVD_RING_RECORD_FLOATS 10
#define AVD_ABI_VERSION 5

typedef enum avd_status {
    AVD_OK = 0,
    AVD_ERR_INVALID_ARG = -1,   /* -> ValueError   */
    AVD_ERR_CUDA = -2,          /* -> RuntimeError */
    AVD_ERR_UNSUPPORTED = -3,   /* -> NotImplementedError */
    AVD_ERR_NO_DEVICE = -4      /* -> RuntimeError: no CUDA device / wrong architecture */
} avd_status;

/* purposes of the Philox4x32-10 counter-based streams (counter word 3) */
enum {
    AVD_RNG_RESET_VEHICLE = 0,
    AVD_RNG_RESET_PLATOON = 1,
    AVD_RNG_OU = 2,
    AVD_RNG_LEADER_EXOG = 3,
    AVD_RNG_REPLAY = 4,
    AVD_RNG_INIT = 5
};

/* ---- environment parameters: the Config scalars the hot path reads (src/config.py:41-104),
 *      plus per-follower system matrices (Vehicle.set_system_matrices, src/environment.py:390-451). */
typedef struct avd_env_params {
    int32_t M;               /* followers per platoon, 1..AVD_MAX_FOLLOWERS (config.pl_size)        */
    int32_t num_states;      /* 4 = Model B, 3 = Model A (environment.py:47-52)                     */
    int32_t model_a;         /* 1: exogenous input = predecessor's post-update accel (env.py:263-267) */
    int32_t can_terminate;   /* config.can_terminate (environment.py:505)                           */
    int32_t centralized;     /* 1: platoon reward = mean over followers (environment.py:234-236)   */
    int32_t rand_uniform;    /* 1: reset draws U(-v,v) instead of N(0,v) (util.py:66-70)            */
    int32_t reset_mode;      /* 0 random (rand_states), 1 fixed maxima, 2 evaluator states (env.py:534-555) */
    int32_t steps_per_episode; /* config.steps_per_episode; 0 = never time out (auto-reset only)    */
    float T, h;              /* sample_rate, timegap                                                 */
    float max_ep, max_ev;    /* terminal thresholds                                                  */
    float action_high, action_low;
    float rew_ep, rew_ev, rew_u, rew_jerk; /* reward coefficients a,b,c,d                           */
    float re_scalar, terminal_reward;
    float reset_ep, reset_ev, reset_a;     /* bounds / std-devs / fixed values selected by reset_mode */
    float reset_leader_a, reset_u;         /* pl_leader_reset_a, reset_max_u                          */
    float ou_theta, ou_dt, ou_sigma, ou_mean; /* OUActionNoise (src/noise.py:3-29)                   */
    float A[AVD_MAX_FOLLOWERS][16];        /* row-major 4x4 per follower                             */
    float B[AVD_MAX_FOLLOWERS][4];
    float C[AVD_MAX_FOLLOWERS][4];
} avd_env_params;

/* ---- device-resident counters, so a captured CUDA graph can be replayed without new arguments */
typedef struct avd_clock {
    uint64_t step_tick;      /* env steps taken (keys OU / leader-exog streams)                      */
    uint64_t ring_count;     /* transitions added per ring == ReplayBuffer.buffer_counter            */
    uint64_t update_tick;    /* learn() calls (keys the replay sampling stream)                      */
    uint64_t reserved;
} avd_clock;

/* ---- a batch of independent training runs.  The batch's P platoons are `runs` contiguous blocks of `platoons_per_run`:
 * platoon p belongs to run s = p / platoons_per_run and draws the streams of platoon p mod platoons_per_run under seed[s]; ring
 * m*P + p draws those of ring m*platoons_per_run + p mod platoons_per_run.  These are the keys a stand-alone run with
 * random_seed = seed[s] uses, so run s of the batch reproduces it.  The struct itself is host memory: every entry that takes
 * one checks runs * platoons_per_run == P and passes it to its kernels by value, so a captured CUDA graph replays it; the
 * seeds (and the optional per-run OU parameters) it points to live in device memory.                                     */
typedef struct avd_runs {
    const uint64_t* seed;      /* [runs] DEVICE pointer: random_seed of every run                             */
    int64_t platoons_per_run;  /* >= 1                                                                       */
    int32_t runs;              /* >= 1                                                                       */
    int32_t reserved;
    const float* ou_sigma;     /* [runs] nullable DEVICE pointer: OU std_dev of every run (NULL: avd_env_params.ou_sigma)  */
    const float* ou_theta;     /* [runs] nullable DEVICE pointer: OU theta of every run (NULL: avd_env_params.ou_theta)    */
} avd_runs;

/* ---- buffers of one shard of platoons (all device pointers; nullable ones are marked) */
typedef struct avd_env_io {
    int64_t P;                 /* platoons in this shard                                             */
    int64_t platoon_id_base;   /* global id of local platoon 0: RNG streams do not depend on sharding */
    uint64_t seed;             /* config.random_seed                                                 */
    const float* x_in;         /* [4][M][P] state before the step                                    */
    float* x_out;              /* [4][M][P] state after the step (ping-pong: never aliases x_in)     */
    float* prev_a;             /* [M][P]   prev_x[2]  (in/out)                                       */
    float* cum_accel;          /* [M][P]   nullable: kinematic observables off                       */
    const float* action_mu;    /* [M][P]   actor output or injected action                           */
    float* ou_state;           /* [M][P]   nullable: no exploration noise (evaluator path)           */
    float* action_out;         /* [M][P]   nullable: clipped action actually applied                 */
    const float* leader_exog;  /* [P]      nullable: see gen_exog                                    */
    float* front_u;            /* [P]      platoon.front_u (used when leader_exog==NULL && !gen_exog) */
    float* front_accel;        /* [P]      platoon.front_accel (Model A fallback)                    */
    float* reward;             /* [M][P]   (centralized: [P]) NEGATED reward as Vehicle.step returns */
    uint8_t* done;             /* [P]      bit0: any follower terminal (platoon_done, environment.py:238);
                                           bit1: episode time limit reached (steps_per_episode)      */
    float* jerk;               /* [M][P]   nullable                                                  */
    float* velocity;           /* [M][P]   nullable (needs cum_accel)                                */
    float* headway;            /* [M][P]   nullable (needs cum_accel)                                */
    float* ring;               /* nullable: replay ring [capacity][M][P][10]                         */
    int64_t ring_capacity;
    int32_t* episode;          /* [P] nullable: per-platoon episode counter (needed for auto_reset)  */
    int32_t* step_in_episode;  /* [P] nullable                                                       */
    float* ep_reward;          /* [M][P] nullable: episodic reward accumulators (trainer.py:321)     */
    float* stats;              /* nullable: += [0..M-1] sum over platoons of reward, [M] #terminal platoons */
    const avd_clock* clock;    /* device clock (step_tick, ring_count)                               */
    int32_t gen_exog;          /* 1: draw leader exog ~ reset_u * N(0,1) on device (trainer.py:292-295) */
    int32_t auto_reset;        /* 1: platoons that are done / timed out are reset inside the kernel  */
    int32_t clip_actions;      /* 1: clip the (noisy) action to [action_low, action_high] (ddpgagent.py:27);
                                  0: apply action_mu as given, like Platoon.step does                 */
    int32_t ep_hist_window;    /* entries of ep_hist per agent (config.weighted_window); 0 with ep_hist == NULL */
    /* End of an episode (avd_env_reset of a platoon that has stepped, or the in-kernel auto-reset): ep_reward is published to
     * last_ep_reward and to slot (finished episode index % ep_hist_window) of ep_hist, then zeroed -- the reference's
     * all_ep_reward_lists[p][m][-weighted_window:] (trainer.py:385-398, 510-517) without leaving the device.              */
    float* last_ep_reward;     /* [M][P] nullable: cumulative reward of the last FINISHED episode              */
    float* ep_hist;            /* [ep_hist_window][M][P] nullable: ring of the last finished episodes' rewards */
    const avd_runs* runs;      /* nullable HOST pointer: the platoons are several runs with their own seeds (seed is then
                                  unused, platoon_id_base must be 0, runs->runs * runs->platoons_per_run must equal P);
                                  NULL: one run keyed by (seed, platoon_id_base + p)                                         */
} avd_env_io;

/* ---- library ------------------------------------------------------------------------------- */
int avd_abi_version(void);
const char* avd_last_error(void);
/* number of CUDA kernels this library has launched in the calling process so far (every launch site counts itself);
 * callers difference it around a region, e.g. bench.py's "gpu_launches" */
int64_t avd_kernel_launches(void);
/* sizeof of the ABI structs as compiled (0 avd_env_params, 1 avd_env_io, 2 avd_clock, 3 avd_net_dims, 4 avd_learn_io,
 * 5 avd_peer_comm, 6 avd_fed_apply_io, 7 avd_runs): bindings assert their own layout against these at load time. */
int64_t avd_sizeof(int which);
/* SM count, compute capability major*10+minor of the current device; AVD_ERR_NO_DEVICE if none */
int avd_device_info(int* sm_count, int* cc, int64_t* total_mem);

/* ---- clock --------------------------------------------------------------------------------- */
/* clock[0] += (d_step, d_ring, d_update): one tiny kernel so it can live inside a CUDA graph.    */
int avd_clock_advance(avd_clock* clock_dev, uint32_t d_step, uint32_t d_ring, uint32_t d_update, void* stream);

/* ---- environment --------------------------------------------------------------------------- */
/* Vehicle.set_system_matrices (environment.py:390-451): fills prm->A/B/C (and prm->T, prm->h) for
 * prm->M followers, computed in double and rounded once to binary32.  method: 0 euler, 1 exact.
 * tau_lead of follower 0 is pl_leader_tau, of the others dyn_coeff (environment.py:57,61).        */
int avd_env_build_matrices(avd_env_params* prm, int method, double sample_rate, double timegap,
                           double dyn_coeff, double pl_leader_tau);

/* Platoon.reset + Vehicle.reset (environment.py:284-301, 520-559) for every platoon with
 * mask[p]!=0 (mask==NULL: all).  Writes x_out AND x_in's accel plane is untouched; prev_a, cum_accel,
 * front_u, front_accel, step_in_episode are reinitialised, episode[p] is incremented afterwards.
 * Random draws: Philox stream (AVD_RNG_RESET_*, id, tick = episode[p]).                           */
int avd_env_reset(const avd_env_params* prm, const avd_env_io* io, const uint8_t* mask, void* stream);

/* Platoon.step (environment.py:209-241) for P platoons, fused with, when the pointers are given:
 * OUActionNoise.__call__ + policy clip (noise.py:14-23, ddpgagent.py:18-29), the leader-exog draw
 * (trainer.py:292-295), ReplayBuffer.add for every (p,m) (replaybuffer.py:37-47), episodic reward
 * accumulation (trainer.py:321) and per-platoon auto-reset.                                        */
int avd_env_step(const avd_env_params* prm, const avd_env_io* io, void* stream);

/* OUActionNoise.__call__ (src/noise.py:14-23) for n independent processes: state[i] is advanced in place
 * with the Philox stream (AVD_RNG_OU, id_base+i, tick) and the new sample is also written to out[i]
 * (out may be NULL).  This is the stand-alone form; avd_env_step fuses the same arithmetic.           */
int avd_ou_sample(const avd_env_params* prm, float* state, float* out, int64_t n, uint64_t id_base,
                  uint64_t seed, uint32_t tick, void* stream);

/* Same step through HOST buffers (the call a drop-in Platoon.step makes): copies actions[M][P]
 * (+ leader_exog[P] if non-NULL) to the device, runs avd_env_step on `io` (whose action_mu /
 * leader_exog must point at device staging of the right size), copies obs (x_out, 4*M*P floats),
 * reward and done back, and synchronises the stream.                                              */
int avd_env_step_host(const avd_env_params* prm, const avd_env_io* io, const float* actions_host,
                      const float* leader_exog_host, float* obs_host, float* reward_host,
                      uint8_t* done_host, void* stream);

/* ---- replay buffer ------------------------------------------------------------------------- */
/* ReplayBuffer.add (replaybuffer.py:37-47) for all M*P rings at once from explicit tuples
 * (the fused path writes the ring from avd_env_step instead).  s, s2: [4][M][P]; a, r: [M][P].   */
int avd_replay_add(float* ring, int64_t capacity, int64_t M, int64_t P, const avd_clock* clock,
                   const float* s, const float* a, const float* r, const float* s2, void* stream);

/* ReplayBuffer.sample index draw (replaybuffer.py:52-54): idx[ring][j] uniform in
 * [0, min(ring_count, capacity)), Philox stream (AVD_RNG_REPLAY, ring_id_base+ring, update_tick).
 * idx_out: int64 [n_rings][batch].                                                                */
int avd_replay_sample_indices(int64_t* idx_out, int64_t n_rings, int64_t ring_id_base, int32_t batch,
                              int64_t capacity, uint64_t seed, const avd_clock* clock, void* stream);

/* ReplayBuffer.sample gathers (replaybuffer.py:57-61): rows are ordered [ring][j]; ring r is
 * (m = r / P ... see layout) -- ring id = m*P + p.  Outputs row-major: s[n][4], a[n], r[n], s2[n][4]. */
int avd_replay_gather(const float* ring, int64_t capacity, int64_t M, int64_t P, const int64_t* idx,
                      int32_t batch, float* s, float* a, float* r, float* s2, void* stream);

/* ReplayBuffer.sample in ONE launch (replaybuffer.py:52-61): the index draw of avd_replay_sample_indices and the gathers of
 * avd_replay_gather, identical results.  A thread owns one Philox block = four samples of a ring and has their twenty 8-byte loads in
 * flight at once (random 40-byte records out of a ring that can span tens of GB: the gather is latency / TLB bound), and the indices
 * need not travel through HBM.  idx_out: nullable int64 [n_rings][batch] (written when the caller wants the draws).                  */
int avd_replay_sample(const float* ring, int64_t capacity, int64_t M, int64_t P, int64_t ring_id_base, int32_t batch, uint64_t seed,
                      const avd_clock* clock, int64_t* idx_out, float* s, float* a, float* r, float* s2, void* stream);

/* The two entries above for a batch of runs (avd_runs, a host pointer): the same kernels, with every ring's Philox stream keyed by
 * its run's seed and its ring id inside the run instead of (seed, ring_id_base + ring).  P (for the index draw: n_rings / M) must be
 * runs * platoons_per_run; AVD_ERR_INVALID_ARG otherwise.                                                                          */
int avd_replay_sample_indices_runs(int64_t* idx_out, int64_t n_rings, int32_t batch, int64_t capacity, const avd_runs* runs,
                                   const avd_clock* clock, void* stream);
int avd_replay_sample_runs(const float* ring, int64_t capacity, int64_t M, int64_t P, int32_t batch, const avd_runs* runs,
                           const avd_clock* clock, int64_t* idx_out, float* s, float* a, float* r, float* s2, void* stream);

/* Fill the whole ring with synthetic transitions (benchmark warm start: steady-state sampling
 * range without running `capacity` env steps).                                                    */
int avd_replay_fill_synthetic(float* ring, int64_t capacity, int64_t M, int64_t P, uint64_t seed, void* stream);

/* ---- DDPG agents ----------------------------------------------------------------------------
 * A population of `A` agents, each with its own actor / critic / target networks (agent/model.py:4-85),
 * Adam state (workers/trainer.py:138-139) and `rows_per_agent` sampled transitions per update.
 * Parameters of one net are one flat fp32 vector per agent, trainable tensors first:
 *   actor  : W1[ns,l1] b1 g1 be1 | W2[l1,l2] b2 g2 be2 | W3[l2,1] b3 || mu1 var1 mu2 var2
 *   critic : Ws[ns,l1] bs Wa[1,la] ba gs bes ga bea | W2[l1+la,l2] b2 g2 be2 | W3[l2,1] b3 || mus vars mua vara mu2 var2
 * (g/be = BatchNormalization gamma/beta, mu/var = its frozen moving statistics; `||` separates the
 * trainable prefix -- the order of Keras `trainable_variables` -- from the non-trainable tail.  The Python
 * mirror exposes views in Keras `.weights` order.)  Dense kernels are row-major [in, out] like Keras.      */
typedef struct avd_net_dims {
    int32_t ns;   /* state width: 4 (Model B) or 3 (Model A)              */
    int32_t l1;   /* actor_layer1_size == critic_layer1_size (256)        */
    int32_t la;   /* critic_act_layer_size (48)                           */
    int32_t l2;   /* actor_layer2_size == critic_layer2_size (128)        */
} avd_net_dims;

typedef struct avd_learn_io {
    avd_net_dims dims;
    int32_t A;                  /* agents                                                              */
    int32_t apply_updates;      /* 1: Adam x2 + Polyak after the gradients (trainer.py:345-356); 0: gradients only */
    int64_t rows_per_agent;     /* transitions per agent and update (reference: batch_size = 64)       */
    float gamma, action_high, tau, actor_lr, critic_lr;
    float adam_beta1, adam_beta2, adam_eps;
    const float* s;             /* [A*rows][s_stride]  sampled states: the first dims.ns words of every row are read     */
    const float* a;             /* [A*rows]                                                            */
    const float* r;             /* [A*rows]                                                            */
    const float* s2;            /* [A*rows][s_stride]                                                  */
    float* actor;               /* [A][actor_total]                                                    */
    float* critic;              /* [A][critic_total]                                                   */
    float* t_actor;
    float* t_critic;
    float* actor_grad;          /* [A][actor_trainable]   out                                          */
    float* critic_grad;         /* [A][critic_trainable]  out                                          */
    float* actor_m; float* actor_v; float* critic_m; float* critic_v;   /* Adam moments, trainable sizes */
    int32_t* actor_t; int32_t* critic_t;                                  /* [A] Adam step counters       */
    const uint8_t* apply_mask;  /* [A] nullable: agents with 0 keep their weights (intrafrl "leader is king") */
    float* loss;                /* [A][2] nullable: critic_loss, actor_loss                            */
    void* workspace;            /* avd_ddpg_workspace_bytes(dims, A, rows_per_agent, precision) bytes  */
    int64_t workspace_bytes;
    int32_t precision;          /* 0: fp32 SIMT kernels (parity mode); 1: bf16 tcgen05 tensor-core GEMMs; 2: fp16 tcgen05;
                                   3: tcgen05 on three-way split bf16 operands, fp32-accurate (avd_gemm_bf16x3; DESIGN.md 4) */
    int32_t s_stride;           /* row pitch of s / s2 in floats: 4 for the replay gather output (avd_replay_gather), 0 = dims.ns */
    const float* agent_hp;      /* [A][4] nullable DEVICE pointer: (gamma, actor_lr, critic_lr, tau) of every agent, used in place of
                                   the scalars above with the same arithmetic (a sweep of hyperparameters in one batch); NULL: the scalars */
} avd_learn_io;

/* sizes of the flat parameter vectors: out4 = {actor_trainable, actor_total, critic_trainable, critic_total} */
int avd_ddpg_param_counts(const avd_net_dims* dims, int64_t* out4);
int64_t avd_ddpg_workspace_bytes(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, int32_t precision);
/* workspace of avd_actor_forward (critic = 0) / avd_critic_forward (critic = 1) for A agents x rows_per_agent rows; -1 on bad arguments */
int64_t avd_forward_workspace_bytes(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, int32_t critic, int32_t precision);

/* Trainer.learn (workers/trainer.py:472-508) for all agents at once: TD target from the target nets,
 * critic MSE gradient, actor -mean(Q) gradient (both on the pre-update weights); then, if apply_updates,
 * tf.keras Adam on both nets (trainer.py:348-349) and ddpgagent.update_target (agent/ddpgagent.py:31-55). */
int avd_ddpg_learn(const avd_learn_io* io, void* stream);

/* actor(state) for `rows_per_agent` rows per agent (trainer.py:287-289 batched).  s element (row n, k) is read
 * at s[n*s_row_stride + k*s_col_stride] so the env's native [4][M][P] state can be fed without a transpose
 * (row stride 1, column stride M*P).  out[n] = action_high * tanh(.)                                    */
int avd_actor_forward(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, const float* actor_params,
                      const float* s, int64_t s_row_stride, int64_t s_col_stride, float action_high, float* out,
                      void* workspace, int64_t workspace_bytes, int32_t precision, void* stream);

/* critic([state, action]) -> q[n] (row-major s[n][ns], a[n]); used by tests and the evaluator. */
int avd_critic_forward(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, const float* critic_params,
                       const float* s, const float* a, float* q, void* workspace, int64_t workspace_bytes,
                       int32_t precision, void* stream);

/* tf.keras.optimizers.Adam.apply_gradients for [A][n] trainable prefixes of [A][stride] parameter vectors:
 * t = ++step[a];  lr_t = lr*sqrt(1-b2^t)/(1-b1^t);  m += (g-m)(1-b1);  v += (g*g-v)(1-b2);
 * theta -= lr_t*m/(sqrt(v)+eps).  grad_agent_stride = n for per-agent gradients, 0 to apply ONE shared
 * gradient vector to every agent (FedAvg'd gradients, trainer.py:419-425).                              */
int avd_adam_apply(float* params, int64_t param_stride, const float* grads, int64_t grad_agent_stride, float* m,
                   float* v, int32_t* step, const uint8_t* apply_mask, int32_t A, int64_t n, float lr, float beta1,
                   float beta2, float eps, void* stream);

/* avd_adam_apply for both nets followed by avd_polyak_update of both targets (trainer.py:348-356), fused: one pass per net
 * applies Adam to the trainable prefix and the Polyak update to ALL weights, then both step counters advance.  Per-agent
 * gradient vectors have stride *_gstride (0 = one shared vector for every agent, as after FedAvg).  agent_hp: nullable [A][4]
 * device table laid out as avd_learn_io.agent_hp; agent a then takes its actor_lr, critic_lr and tau from row a.              */
int avd_adam_polyak_apply2(float* actor, float* t_actor, int64_t actor_total, const float* actor_grad, int64_t actor_gstride,
                           float* actor_m, float* actor_v, int32_t* actor_step, int64_t actor_train, float actor_lr, float* critic,
                           float* t_critic, int64_t critic_total, const float* critic_grad, int64_t critic_gstride, float* critic_m,
                           float* critic_v, int32_t* critic_step, int64_t critic_train, float critic_lr, const uint8_t* apply_mask,
                           int32_t A, float beta1, float beta2, float eps, float tau, const float* agent_hp, void* stream);

/* ddpgagent.update_target (agent/ddpgagent.py:44-55): target = tau*online + (1-tau)*target over n floats
 * per agent (ALL weights incl. BN statistics).                                                          */
int avd_polyak_update(float* target, const float* online, const uint8_t* apply_mask, int32_t A, int64_t n, float tau,
                      void* stream);

/* federated.Server.get_avg_params / get_weighted_avg_params (src/server/federated.py:18-122) for flat
 * vectors: out[s][j] = scale[s] * sum_x weight[s][x] * in[member(s,x)][j].  Members of system s are
 * in[(s*member_stride_s + x*member_stride_x)] rows of length n (row pitch `pitch`); weights NULL = 1;
 * scale NULL = 1/X (plain mean).  One launch; used locally before / after the NCCL allreduce.           */
int avd_fed_reduce(float* out, int64_t out_pitch, const float* in, int64_t pitch, int32_t n_systems, int32_t n_members,
                   int64_t member_stride_s, int64_t member_stride_x, const float* weights, const float* scale, int64_t n,
                   void* stream);

/* One-launch forms for a whole federated round (actor and critic vectors side by side in one [systems][pitch] buffer):
 * avd_fed_reduce2: out[s][0..na) / out[s][na..na+nc) = sum_x w[s][x] * actor / critic vector of member (s, x) (weights NULL = 1)
 * and out[s][na+nc] = sum_x w[s][x] -- the divisor that travels through the exchange; avd_fed_broadcast2: the way back.      */
int avd_fed_reduce2(float* out, int64_t out_pitch, const float* in_a, int64_t pitch_a, int64_t na, const float* in_c, int64_t pitch_c,
                    int64_t nc, int32_t n_systems, int32_t n_members, int64_t member_stride_s, int64_t member_stride_x,
                    const float* weights, void* stream);
int avd_fed_broadcast2(float* out_a, int64_t pitch_a, int64_t na, float* out_c, int64_t pitch_c, int64_t nc, const float* in,
                       int64_t in_pitch, int32_t n_systems, int32_t n_members, int64_t member_stride_s, int64_t member_stride_x,
                       const uint8_t* apply_mask, void* stream);

/* Trainer.get_weight (workers/trainer.py:385-398) for all agents: w = |1 / mean(last `window` episodic rewards)| from the ring of
 * finished-episode rewards the env kernel keeps (avd_env_io.ep_hist, [window][M][P], P = G*E; an agent's episodic reward is the mean
 * over its group's E platoons).  out_w[m*G + g] (interfrl: systems = followers) or, with transpose, out_w[g*M + m] (intrafrl).       */
int avd_fed_weights_from_history(const float* ep_hist, int32_t window, int32_t M, int64_t G, int64_t E, float* out_w,
                                 int32_t transpose, void* stream);

/* buf[s][0..n) *= 1 / buf[s][n]: turns the exchanged (weighted) sums into means (federated.py:62 / :110); the
 * divisor (member count or sum of weights) travels in column n of the same buffer through the all_reduce.     */
int avd_fed_finalize(float* buf, int64_t pitch, int32_t n_systems, int64_t n, void* stream);

/* NVLink-native exchange step of an interfrl round (replaces ncclAllReduce + avd_fed_finalize; src/server/federated.py:56-62,
 * 109-110 across GPUs).  Every rank owns one allocation of a SYMMETRIC buffer (peer-mapped into all ranks, e.g. from
 * torch.distributed._symmetric_memory); peer_base[r] is rank r's allocation as seen from this process, multicast_base the NVLS
 * multicast mapping of the same allocation (0 if the fabric has none).  Inside the allocation: `flag_offset` -> AVD_MAX_PEERS
 * uint32 epoch flags (zero-initialised once), `data_offset` -> this round's partial sums [n_systems][pitch] fp32 with the local
 * member count / weight sum in column n.  The kernel signals the round's epoch to every peer, waits for all peers, reads the sums
 * over ranks (multimem.ld_reduce in the NVSwitch, or peer loads) and writes out[s][j] = sum_r data_r[s][j] / sum_r data_r[s][n]
 * for j < n and the reduced divisor itself to out[s][n] (fed_weight_sums, trainer.py:358-359).
 * `ctrl`: FOUR zero-initialised uint32 words in LOCAL device memory, owned by the exchange kernels: [0] counts the completed rounds
 * (the epoch: it is read at kernel start and advanced by the round's last CTA, so nothing about the barrier is baked into launch
 * arguments and a captured CUDA graph replays correctly), [1] is a CTA ticket, [2] stays 0 unless a peer's signal did not arrive within
 * the barrier's time limit (environment AVD_PEER_TIMEOUT_MS, default 20000): then it holds 1 + that peer's rank, the round's results
 * are undefined and the caller must treat the exchange as failed (the kernel gives up instead of spinning forever), [3] reserved.
 * Every rank must issue the same sequence of
 * exchange calls (this entry and avd_fed_apply_gradients share the epoch); the caller alternates `data_offset` between two halves. */
#define AVD_MAX_PEERS 16
typedef struct avd_peer_comm {
    int32_t rank, world;
    uint32_t reserved0, reserved1;
    uint64_t peer_base[AVD_MAX_PEERS];
    uint64_t multicast_base;
} avd_peer_comm;
int avd_fed_exchange_peer(const avd_peer_comm* comm, int64_t flag_offset, int64_t data_offset, uint32_t* ctrl, float* out,
                          int64_t pitch, int32_t n_systems, int64_t n, void* stream);

/* One federated GRADIENTS round after avd_fed_reduce2 (train_all_models_federated_gradients, workers/trainer.py:400-431), fused:
 * cross-rank barrier -> sums over ranks (NVLS multimem.ld_reduce / peer loads; world == 1: `local_sums`) -> division by the reduced
 * member count / weight sum (federated.py:62, :110) -> for every local member (s, x) = agent s*member_stride_s + x*member_stride_x
 * with apply_mask != 0: tf.keras Adam on the trainable prefix with the averaged gradient, Polyak update of ALL target weights
 * (ddpgagent.py:44-55), Adam step counters += 1.  The partial sums are rows [n_systems][pitch] with the actor gradient in columns
 * [0, actor_train), the critic gradient in [actor_train, actor_train + critic_train) and the divisor in the next column.
 * *_grad_out (nullable): the averaged gradient is also stored into every member's gradient row.  wsum_out (nullable): [n_systems]
 * reduced divisors.  `ctrl`: see avd_fed_exchange_peer.                                                                          */
typedef struct avd_fed_apply_io {
    avd_peer_comm comm;
    int64_t flag_offset, data_offset;
    const float* local_sums;      /* world == 1 only: [n_systems][pitch]                               */
    uint32_t* ctrl;
    int64_t pitch;
    int32_t n_systems, n_members;
    int64_t member_stride_s, member_stride_x;
    int32_t A, reserved0;
    float *actor, *t_actor, *actor_m, *actor_v; int32_t* actor_step; float* actor_grad_out;
    int64_t actor_total, actor_train;
    float *critic, *t_critic, *critic_m, *critic_v; int32_t* critic_step; float* critic_grad_out;
    int64_t critic_total, critic_train;
    const uint8_t* apply_mask;    /* [A] nullable                                                      */
    float* wsum_out;
    float actor_lr, critic_lr, beta1, beta2, eps, tau;
    const float* agent_hp;        /* [A][4] nullable: per-agent (gamma, actor_lr, critic_lr, tau) as avd_learn_io.agent_hp; the
                                     learning rates and tau are read.  A <= 25,600 without it, A <= 17,066 with it (shared memory) */
} avd_fed_apply_io;
int avd_fed_apply_gradients(const avd_fed_apply_io* io, void* stream);

/* out[a][j] = in[src(a)][j]: broadcast system averages back onto members (set_weights, trainer.py:448-456). */
int avd_fed_broadcast(float* out, int64_t out_pitch, const float* in, int64_t in_pitch, int32_t n_systems,
                      int32_t n_members, int64_t member_stride_s, int64_t member_stride_x, const uint8_t* apply_mask,
                      int64_t n, void* stream);

/* ---- tensor-core GEMM (tcgen05 + TMEM + TMA), the building block of precision = 1 ------------------
 * C[b] (fp32, M x N, row pitch ldc) = / += op(A[b]) op(B[b]) with bf16 operands and fp32 accumulation.
 *   layout 0 (TN: forward, dgrad): A[b] is [M][K] (pitch lda), B[b] is [N][K] (pitch ldb); C = A B^T; splitk>1 accumulates
 *                                  atomically into C (caller zeroes it).
 *   layout 1 (NT: wgrad)         : A[b] is [K][M], B[b] is [K][N]; C += A^T B, always accumulated atomically (the
 *                                  contraction runs over batch rows and is split over `splitk` CTAs).
 * Pitches and batch strides are in elements and must be multiples of 8; operands 16-byte aligned.
 * Replaces the Dense(256->128) / Dense(304->128) matmuls and their gradients inside Trainer.learn
 * (workers/trainer.py:492-506 via agent/model.py:30,74).                                                  */
int avd_gemm_bf16(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B,
                  int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, void* stream);

/* Same GEMM with fp16 (a_fmt = b_fmt = 0) or bf16 (1) operands.  Mixed formats return AVD_ERR_UNSUPPORTED: the tcgen05 instruction
 * descriptor has a format field per operand, but B200 traps on fp16 x bf16.                                                         */
int avd_gemm_f16kind(int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B,
                     int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, int a_fmt, int b_fmt, void* stream);

/* The same GEMM on fp32-accurate split operands, the building block of precision = 3: every operand element x is given as three bf16
 * planes hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid) (24 significand bits together), stored [plane][batch][rows][inner]:
 * plane p of batch b starts at A_planes + (p * batch + b) * a_batch (likewise B), so a_batch / b_batch must be positive.  Each K block
 * runs the six products hi.hi + hi.mid + mid.hi + hi.lo + mid.mid + lo.hi into one fp32 accumulator; the dropped ones are below
 * 2^-27 |a||b|.  Layouts, pitches, split-K and alignment as avd_gemm_bf16.                                                         */
int avd_gemm_bf16x3(int layout, int batch, int M, int N, int K, const void* A_planes, int64_t lda, int64_t a_batch, const void* B_planes,
                    int64_t ldb, int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, void* stream);

/* ---- raw RNG access (parity tests: bit-exact against oracle/philox_np.py) ------------------- */
int avd_rng_words(uint32_t* out4 /*[n][4]*/, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose,
                  uint64_t seed, void* stream);
int avd_rng_normals(float* out4 /*[n][4]*/, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose,
                    uint64_t seed, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVDDPG_B200_H */
