"""Host-side mirror of the reference's ``src/environment.py`` over the CUDA platoon kernels.

``BatchedPlatoons`` is the real thing: P independent platoons of M followers resident in HBM, stepped by
one kernel launch (csrc/avd_env.cu) through the C ABI.  ``Platoon`` and ``Vehicle`` are drop-in shims with
the reference's constructor signatures, attributes and return conventions
(/root/reference/src/environment.py:8-85, 209-301, 304-559) -- each is a view onto a 1-platoon batch, so
``workers/trainer.py`` / ``workers/evaluator.py`` style code runs unchanged.

No CPU fallback exists: constructing any of these without the shared library or a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .config import env_params_from_config


class DeviceClock:
    """avd_clock in device memory (step_tick, ring_count, update_tick): kernels read it, a one-thread
    kernel advances it, so a CUDA graph of the training step can be replayed with no new arguments."""

    def __init__(self, device):
        self.t = torch.zeros(4, dtype=torch.int64, device=device)

    @property
    def ptr(self):
        return C.c_void_p(self.t.data_ptr())

    def advance(self, step=0, ring=0, update=0):
        _lib.check(_lib.load().avd_clock_advance(self.ptr, step, ring, update, _lib.current_stream()))

    def set(self, step_tick=None, ring_count=None, update_tick=None):
        vals = self.t.tolist()
        for i, v in enumerate((step_tick, ring_count, update_tick)):
            if v is not None:
                vals[i] = int(v)
        self.t.copy_(torch.tensor(vals, dtype=torch.int64))

    def read(self):
        s, r, u, _ = self.t.tolist()
        return {"step_tick": s, "ring_count": r, "update_tick": u}


class RunTable:
    """S independent training runs that share one batch of P = S * platoons_per_run platoons (avd_runs: a host struct the library
    checks and hands to its kernels by value, over a device array of the seeds, so a captured CUDA graph replays it).  Run s owns
    platoons [s * Pr, (s + 1) * Pr) and draws every random stream of the stand-alone run with random_seed = seeds[s]: its platoon
    p' is keyed (seeds[s], p') and its ring m * Pr + p' likewise.  ou_sigma / ou_theta: optional per-run OU std_dev / theta (one value
    per seed) in place of the configuration's, for a hyperparameter sweep; None keeps the configuration's value for every run."""

    def __init__(self, seeds, platoons_per_run: int, device, ou_sigma=None, ou_theta=None):
        seeds = [int(k) for k in seeds]
        if not seeds:
            raise ValueError("a run table needs at least one seed")
        bad = [k for k in seeds if not 0 <= k < 1 << 64]
        if bad:
            raise ValueError(f"seeds must be unsigned 64-bit integers, got {bad}")
        if int(platoons_per_run) < 1:
            raise ValueError("platoons_per_run must be positive")
        self.seeds, self.S, self.Pr = seeds, len(seeds), int(platoons_per_run)
        # uint64 bit patterns in an int64 tensor (the kernels read them as uint64_t)
        self.seed_t = torch.tensor([k - (1 << 64) if k >= 1 << 63 else k for k in seeds], dtype=torch.int64, device=device)
        self.table = _lib.Runs()
        self.table.seed, self.table.platoons_per_run, self.table.runs = self.seed_t.data_ptr(), self.Pr, self.S
        self.ou_sigma = self._per_run("ou_sigma", ou_sigma, device)
        self.ou_theta = self._per_run("ou_theta", ou_theta, device)
        self.table.ou_sigma = None if self.ou_sigma is None else self.ou_sigma.data_ptr()
        self.table.ou_theta = None if self.ou_theta is None else self.ou_theta.data_ptr()

    def _per_run(self, name, values, device):
        if values is None:
            return None
        values = [float(v) for v in values]
        if len(values) != self.S:
            raise ValueError(f"{name}: {len(values)} values for {self.S} runs")
        return torch.tensor(values, dtype=torch.float32, device=device)

    @property
    def ptr(self):
        return C.c_void_p(C.addressof(self.table))

    @property
    def P(self) -> int:
        return self.S * self.Pr


class BatchedPlatoons:
    """P platoons x M followers on one GPU.

    Layout (see include/avddpg_b200.h): state ``x[f][m][p]`` with the platoon index fastest; every
    tensor returned to the caller is a zero-copy *view* in the reference's logical order
    (``obs[P, M, num_states]``, ``reward[P, M]``, ``done[P]``).  State buffers ping-pong, so a returned
    observation stays valid until the second following ``step`` -- the caller may keep it as
    ``prev_state`` exactly like workers/trainer.py:271 does.
    """

    def __init__(self, num_platoons: int, length: int, config, *, device=None, platoon_id_base: int = 0,
                 seed: Optional[int] = None, rand_states: bool = True, evaluator_states_enabled: bool = False,
                 track_kinematics: bool = True, ring=None, clock: Optional[DeviceClock] = None,
                 steps_per_episode: Optional[int] = None, auto_reset: bool = False, collect_stats: bool = False,
                 track_episodes: bool = True, store_actions: bool = True, reward_history: int = 0,
                 runs: Optional[RunTable] = None):
        """runs: the platoons are runs.S independent runs of runs.Pr platoons each (see RunTable); seed and platoon_id_base are
        then unused."""
        self.lib = _lib.load()
        _lib.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedPlatoons is CUDA-only (no CPU fallback)")
        self.P, self.M, self.config = int(num_platoons), int(length), config
        self.prm = env_params_from_config(config, self.M, rand_states, evaluator_states_enabled, steps_per_episode)
        self.num_states = int(self.prm.num_states)
        self.centralized = bool(self.prm.centralized)
        self.seed = int(getattr(config, "random_seed", 1) if seed is None else seed)
        if runs is not None and (runs.P != self.P or platoon_id_base != 0):
            raise ValueError(f"a run table of {runs.S} x {runs.Pr} platoons needs P = {runs.P} and platoon_id_base = 0")
        self.runs = runs
        P, M, dev = self.P, self.M, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        self._x = torch.zeros(2, 4, M, P, **f32)
        self._cur = 0
        self.prev_a = torch.zeros(M, P, **f32)
        self.cum_accel = torch.zeros(M, P, **f32) if track_kinematics else None
        self.jerk = torch.zeros(M, P, **f32) if track_kinematics else None
        self.velocity = torch.zeros(M, P, **f32) if track_kinematics else None
        self.headway = torch.zeros(M, P, **f32) if track_kinematics else None
        self.ou_state = torch.zeros(M, P, **f32)
        self.action_mu = torch.zeros(M, P, **f32)
        self.action_out = torch.zeros(M, P, **f32) if store_actions else None
        self.leader_exog = torch.zeros(P, **f32)
        self.front_u = torch.zeros(P, **f32)
        self.front_accel = torch.zeros(P, **f32)
        self._reward = torch.zeros((P,) if self.centralized else (M, P), **f32)
        self._done = torch.zeros(P, dtype=torch.uint8, device=dev)
        if auto_reset and not track_episodes:
            raise ValueError("auto_reset needs track_episodes=True")
        self.episode = torch.zeros(P, dtype=torch.int32, device=dev) if track_episodes else None
        self.step_in_episode = torch.zeros(P, dtype=torch.int32, device=dev) if track_episodes else None
        self.ep_reward = torch.zeros(M, P, **f32) if track_episodes else None
        # finished-episode rewards: the last one, and a ring of the last `reward_history` (config.weighted_window) per agent --
        # the device-resident all_ep_reward_lists[p][m][-weighted_window:] of workers/trainer.py:385-398
        self.last_ep_reward = torch.zeros(M, P, **f32) if track_episodes else None
        self.ep_hist = torch.zeros(int(reward_history), M, P, **f32) if (track_episodes and reward_history > 0) else None
        self.stats = torch.zeros(M + 1, **f32) if collect_stats else None
        self.clock = clock if clock is not None else DeviceClock(dev)
        self.ring = ring
        self.auto_reset = bool(auto_reset)
        self.io = _lib.EnvIO()
        io = self.io
        io.P, io.platoon_id_base, io.seed = P, int(platoon_id_base), self.seed
        io.ep_hist_window = 0 if self.ep_hist is None else int(reward_history)
        for name in ("prev_a", "cum_accel", "front_u", "front_accel", "jerk", "velocity", "headway", "episode",
                     "step_in_episode", "ep_reward", "stats", "last_ep_reward", "ep_hist"):
            t = getattr(self, name)
            setattr(io, name, None if t is None else t.data_ptr())
        io.reward, io.done = self._reward.data_ptr(), self._done.data_ptr()
        io.clock = self.clock.t.data_ptr()
        io.runs = None if runs is None else C.addressof(runs.table)
        if ring is not None:
            if ring.M != M or ring.P != P:
                raise ValueError("replay ring shape does not match the platoon batch")
            io.ring, io.ring_capacity = ring.data.data_ptr(), ring.capacity
        self._launches = 0

    # ------------------------------------------------------------------ views
    def _obs_view(self, buf):
        return self._x[buf].permute(2, 1, 0)[..., : self.num_states]

    @property
    def obs(self):
        """Current observation, [P, M, num_states] (view)."""
        return self._obs_view(self._cur)

    @property
    def state(self):
        """Full 4-component state [P, M, 4] (view), like Vehicle.x."""
        return self._x[self._cur].permute(2, 1, 0)

    @property
    def native_state(self):
        """[4, M, P] tensor the kernels read -- feed this to the actor kernels without a transpose."""
        return self._x[self._cur]

    @property
    def reward(self):
        return self._reward.view(self.P, 1) if self.centralized else self._reward.t()

    @property
    def done(self):
        return (self._done & 1).bool()

    @property
    def truncated(self):
        return (self._done & 2).bool()

    @property
    def gpu_launches(self):
        return self._launches

    # ------------------------------------------------------------------ operations
    def set_state(self, x, front_accel=None, front_u=None):
        """Inject states: x[P, M, 3|4] = (ep, ev, a[, a_lead]).  With 3 columns a_lead is chained as
        Platoon.reset does (environment.py:291-294).  prev_x := x, kinematic sums := 0."""
        def dev(v, shape):
            if not torch.is_tensor(v):
                v = np.asarray(v, dtype=np.float32)
            return torch.as_tensor(v, dtype=torch.float32, device=self.device).reshape(shape)

        x = dev(x, (self.P, self.M, -1)) if not torch.is_tensor(x) else x.to(self.device, torch.float32)
        if x.shape[:2] != (self.P, self.M):
            raise ValueError(f"expected [P={self.P}, M={self.M}, 3|4], got {tuple(x.shape)}")
        if front_accel is not None:
            self.front_accel.copy_(dev(front_accel, self.P))
        if front_u is not None:
            self.front_u.copy_(dev(front_u, self.P))
        full = torch.zeros(self.P, self.M, 4, dtype=torch.float32, device=self.device)
        full[..., : x.shape[-1]] = x
        if x.shape[-1] == 3:
            full[:, 0, 3] = self.front_accel
            full[:, 1:, 3] = full[:, :-1, 2]
        self._x[self._cur].copy_(full.permute(2, 1, 0))
        self.prev_a.copy_(self._x[self._cur][2])
        if self.cum_accel is not None:
            self.cum_accel.zero_()
        if self.step_in_episode is not None:
            self.step_in_episode.zero_()
        return self.obs

    def reset(self, mask=None):
        """Platoon.reset for every platoon (or those with mask[p] true).  Returns obs [P, M, ns]."""
        io = self.io
        io.x_in = None
        io.x_out = self._x[self._cur].data_ptr()
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if m.numel() != self.P:
                raise ValueError("mask must have one entry per platoon")
        _lib.check(self.lib.avd_env_reset(C.byref(self.prm), C.byref(io), _lib.ptr(m), _lib.current_stream()))
        self._launches += 1
        return self.obs

    def _prepare(self, explore, clip, leader_exog, gen_exog):
        io = self.io
        io.x_in = self._x[self._cur].data_ptr()
        io.x_out = self._x[self._cur ^ 1].data_ptr()
        io.action_mu = self.action_mu.data_ptr()
        io.ou_state = self.ou_state.data_ptr() if explore else None
        io.action_out = None if self.action_out is None else self.action_out.data_ptr()
        io.clip_actions = int(explore if clip is None else clip)
        io.leader_exog = self.leader_exog.data_ptr() if leader_exog else None
        io.gen_exog = int(gen_exog)
        io.auto_reset = int(self.auto_reset)

    def step_native(self, *, explore=False, clip=None, leader_exog=False, gen_exog=False, advance_clock=True):
        """One launch on whatever is already in ``self.action_mu`` ([M,P]) / ``self.leader_exog`` ([P]).
        The zero-copy path used by the training loop and the benchmark."""
        self._prepare(explore, clip, leader_exog, gen_exog)
        _lib.check(self.lib.avd_env_step(C.byref(self.prm), C.byref(self.io), _lib.current_stream()))
        self._cur ^= 1
        self._launches += 1
        if advance_clock:
            self.clock.advance(step=1, ring=1 if self.ring is not None else 0)
            self._launches += 1

    def step(self, actions, leader_exog=None, *, explore=False, clip=None, gen_exog=False):
        """Platoon.step for the whole batch.  actions: [P, M] (tensor or array); leader_exog: [P], scalar
        or None (None -> platoon.front_u / front_accel, or a fresh N(0, reset_max_u) draw when
        gen_exog=True, as workers/trainer.py:292-295 does).  Returns (obs[P,M,ns], reward[P,M], done[P])."""
        if not torch.is_tensor(actions):
            actions = np.asarray(actions, dtype=np.float32)
        a = torch.as_tensor(actions, dtype=torch.float32, device=self.device).reshape(self.P, self.M)
        self.action_mu.copy_(a.t())
        if leader_exog is not None:
            if not torch.is_tensor(leader_exog):
                leader_exog = np.asarray(leader_exog, dtype=np.float32)
            self.leader_exog.copy_(torch.as_tensor(leader_exog, dtype=torch.float32, device=self.device).reshape(-1).expand(self.P))
        self.step_native(explore=explore, clip=clip, leader_exog=leader_exog is not None, gen_exog=gen_exog)
        return self.obs, self.reward, self.done

    def get_jerk(self):
        if self.jerk is None:
            raise RuntimeError("constructed with track_kinematics=False")
        return self.jerk.t()


# ====================================================================================== drop-in shims
class _FollowerView:
    """followers[i] of a shim Platoon: the attributes trainer/evaluator read (x, u, tau, ...)."""

    def __init__(self, platoon: "Platoon", idx: int):
        self._pl, self.idx = platoon, idx
        conf = platoon.config
        self.tau = conf.dyn_coeff
        self.tau_lead = conf.pl_leader_tau if idx == 0 else conf.dyn_coeff
        self.h, self.T = conf.timegap, conf.sample_rate
        self.stand_still = 8
        prm = platoon._env.prm
        self.A = np.array(list(prm.A[idx]), dtype=np.float64).reshape(4, 4)
        self.B = np.array(list(prm.B[idx]), dtype=np.float64)
        self.C = np.array(list(prm.C[idx]), dtype=np.float64)

    def _scalar(self, tensor):
        return float(tensor[self.idx, 0].item())

    @property
    def x(self):
        return self._pl._env.state[0, self.idx].double().cpu().numpy()

    @property
    def u(self):
        return self._scalar(self._pl._env.action_out)

    @property
    def jerk(self):
        return self._scalar(self._pl._env.jerk)

    @property
    def velocity(self):
        return self._scalar(self._pl._env.velocity)

    @property
    def headway(self):
        return self._scalar(self._pl._env.headway)

    @property
    def desired_headway(self):
        return self.stand_still + self.h * self.velocity

    @property
    def reward(self):
        return -float(self._pl._last_reward[self.idx])


class Platoon:
    """Drop-in for environment.Platoon (src/environment.py:8-301) backed by a 1-platoon GPU batch."""

    def __init__(self, length, config, pl_idx, rand_states=True, evaluator_states_enabled=False, *, seed=None,
                 strict_reference_limits=False):
        if strict_reference_limits and length > 6:   # environment.py:84-85 (rendering colour table)
            raise ValueError(f"Platoon of length {length}, but only have 6! Add more colors in environment to "
                             "work with larger platoons in rendering!")
        self.pl_idx, self.config, self.length = pl_idx, config, length
        self.rand_states, self.evaluator_states_enabled = rand_states, evaluator_states_enabled
        idx = int(pl_idx) if isinstance(pl_idx, (int, np.integer)) else 0
        self._env = BatchedPlatoons(1, length, config, platoon_id_base=idx, seed=seed, rand_states=rand_states,
                                    evaluator_states_enabled=evaluator_states_enabled)
        centralized = config.framework == "centralized"
        self.multiplier = length if centralized else 1                        # environment.py:35-42
        self.hidden_multiplier = config.centrl_hidd_mult if centralized else 1
        self.num_models = 1 if centralized else length
        self.def_num_actions = 1
        self.num_actions = self.def_num_actions * self.multiplier
        self.def_num_states = self._env.num_states
        self.num_states = self.def_num_states * self.multiplier
        self.number_of_reward_components = Vehicle.number_of_reward_components
        self.state_lbs = {0: "$e_{pi,k}$", 1: "$e_{vi,k}$", 2: "$a_{i,k}$", 3: "$a_{i-1,k}$"}
        self.jerk_lb, self.exog_lbl = "jerk", "$u_{i,k}$"
        self.pl_leader_tau = config.pl_leader_tau
        self.viewer = None
        n = length
        self._h_act = torch.zeros(n, dtype=torch.float32).pin_memory()
        self._h_exog = torch.zeros(1, dtype=torch.float32).pin_memory()
        self._h_obs = torch.zeros(4 * n, dtype=torch.float32).pin_memory()
        self._h_rew = torch.zeros(1 if centralized else n, dtype=torch.float32).pin_memory()
        self._h_done = torch.zeros(1, dtype=torch.uint8).pin_memory()
        self._last_reward = np.zeros(n)
        self._env.reset()                       # the reference constructor initialises the states too
        self.followers = [_FollowerView(self, i) for i in range(length)]

    @property
    def front_u(self):
        return float(self._env.front_u.item())

    @property
    def front_accel(self):
        return float(self._env.front_accel.item())

    def _states_out(self, obs_pm):
        rows = [np.asarray(obs_pm[m], dtype=np.float64) for m in range(self.length)]
        if self.config.framework == "centralized":
            return [list(np.concatenate(rows).flat)]
        return rows

    def reset(self):
        obs = self._env.reset().double().cpu().numpy()[0]
        return self._states_out(obs)

    def step(self, actions, leader_exog=None, debug_mode=False):
        """-> (states list[M] of arrays[num_states], rewards list[M], platoon_done bool); one C-ABI call
        with host buffers (avd_env_step_host)."""
        env, M = self._env, self.length
        self._h_act.copy_(torch.as_tensor(np.asarray(actions, dtype=np.float32).reshape(M)))
        exog_ptr = None
        if leader_exog is not None:
            self._h_exog[0] = float(leader_exog)
            exog_ptr = C.c_void_p(self._h_exog.data_ptr())
        env._prepare(False, False, leader_exog is not None, False)
        _lib.check(env.lib.avd_env_step_host(C.byref(env.prm), C.byref(env.io), C.c_void_p(self._h_act.data_ptr()),
                                             exog_ptr, C.c_void_p(self._h_obs.data_ptr()),
                                             C.c_void_p(self._h_rew.data_ptr()), C.c_void_p(self._h_done.data_ptr()),
                                             _lib.current_stream()))
        env._cur ^= 1
        env._launches += 1
        env.clock.advance(step=1)
        obs = self._h_obs.numpy().reshape(4, M).T[:, : env.num_states]
        rew = self._h_rew.numpy().astype(np.float64)
        self._last_reward = rew if len(rew) == M else np.repeat(rew, M)
        return self._states_out(obs), [r for r in rew], bool(self._h_done[0] & 1)

    def get_jerk(self):
        j = self._env.jerk[:, 0].double().cpu().numpy()
        return [[float(v)] for v in j]

    def get_exogenous_info(self, idx, leader_exog):
        if self.config.model == "ModelB":
            if idx == 0:
                return self.front_u if leader_exog is None else leader_exog
            return self.followers[idx - 1].u
        if idx == 0:
            return self.front_accel if leader_exog is None else leader_exog
        return self.followers[idx - 1].x[2]

    def get_reward(self, states, rewards):
        return (1 / self.length) * sum(rewards)

    def render(self, mode="human"):   # GUI is out of scope (SURVEY §2 row 15)
        return None

    def close_render(self):
        self.viewer = None


class Vehicle:
    """Drop-in for environment.Vehicle (src/environment.py:304-559): one follower, exogenous input given
    explicitly.  Backed by a 1x1 batch whose 'leader tau' is this vehicle's tau_lead."""
    number_of_reward_components = 4

    def __init__(self, idx, config, tau_lead=None, a_lead=None, num_states=None, num_actions=None, rand_states=True,
                 evaluator_states_enabled=True, *, seed=None):
        if tau_lead is None:
            raise TypeError("tau_lead is required (the reference fails at environment.py:392 without it)")
        import copy
        conf = copy.copy(config)
        conf.pl_leader_tau = tau_lead
        conf.framework = "decentralized"
        self.config, self.idx = config, idx
        self._env = BatchedPlatoons(1, 1, conf, platoon_id_base=int(idx), seed=seed, rand_states=rand_states,
                                    evaluator_states_enabled=evaluator_states_enabled)
        self.num_states = self._env.num_states if num_states is None else num_states
        self.num_actions = 1
        self.tau, self.tau_lead = config.dyn_coeff, tau_lead
        prm = self._env.prm
        self.A = np.array(list(prm.A[0]), dtype=np.float64).reshape(4, 4)
        self.B = np.array(list(prm.B[0]), dtype=np.float64)
        self.C = np.array(list(prm.C[0]), dtype=np.float64)
        self.u, self.reward = 0.0, 0.0
        self.reset(a_lead)

    @property
    def x(self):
        return self._env.state[0, 0].double().cpu().numpy()

    @property
    def jerk(self):
        return float(self._env.jerk.item())

    @property
    def velocity(self):
        return float(self._env.velocity.item())

    @property
    def headway(self):
        return float(self._env.headway.item())

    def set_state(self, state):
        self._env.set_state(np.asarray(state, dtype=np.float32).reshape(1, 1, -1))

    def reset(self, a_lead=None):
        self._env.reset()
        x = self._env.state[0, 0].clone()
        x[3] = 0.0 if a_lead is None else float(a_lead)
        self._env.set_state(x.reshape(1, 1, 4))
        self.u = 0.0
        return self.x[: self.num_states]

    def step(self, u, exog_info, debug_mode=False):
        obs, rew, done = self._env.step([[float(u)]], float(exog_info))
        self.u = float(u)
        r = float(rew.item())
        self.reward = -r
        return obs[0, 0].double().cpu().numpy()[: self.num_states], r, bool(done.item())
