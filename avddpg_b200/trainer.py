"""The learn / act / update part of the reference's ``workers/trainer.py`` on the GPU.

``DDPGPopulation`` owns the actor, critic, target networks and Adam state of A agents as flat HBM vectors
and runs, for all of them at once,
    act()   : actor(state) for every vehicle (trainer.py:286-289; OU noise + clip are fused into the env step)
    learn() : Trainer.learn (trainer.py:472-508) + Adam x2 + Polyak (trainer.py:345-356) -- one C-ABI call
Agent a = m*G + g is follower m of platoon-group g; its ``rows_per_agent`` sampled transitions are rows
[a*R, (a+1)*R) of the replay gather output, which is exactly the order ReplayRings produces when the
group's platoons are contiguous (ring id = m*P + p, P = G*E).  With E envs per group every agent's update
is the mean gradient over its E per-platoon minibatches of 64 -- the reference's interfrl/gradients round
(trainer.py:400-431) for platoons that share weights, without the E redundant copies of the weights.

``Trainer`` keeps the reference's ``learn(rbuffer, actor, critic, target_actor, target_critic)`` signature for
single-agent model objects from avddpg_b200.model.
"""
from __future__ import annotations

import copy
import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .model import NetBank, dims_from_config


class DDPGPopulation:
    def __init__(self, num_groups: int, num_followers: int, config, *, num_states: int = 4, rows_per_agent: int = 64,
                 device=None, seed: Optional[int] = None, precision: int = 0, seeds: Optional[Sequence[int]] = None,
                 overrides: Optional[Sequence[dict]] = None):
        """seeds: the G groups are len(seeds) independent runs of G / len(seeds) groups each; run s starts from the weights the
        stand-alone population with seed seeds[s] draws (its agents m*G + s*Gr + g', see run_agents).
        overrides: one dict per seed (config.run_configs): run s learns with its own gamma, actor_lr, critic_lr and tau.  They go into
        the per-agent table `hp` [A, 4] = (gamma, actor_lr, critic_lr, tau), which learn() and apply_gradients_and_soft_update()
        (and so FederatedAggregator) use in place of the config scalars; without overrides `hp` is None."""
        self.lib = _lib.load()
        _lib.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.G, self.M, self.A = int(num_groups), int(num_followers), int(num_groups) * int(num_followers)
        self.config, self.R, self.precision = config, int(rows_per_agent), int(precision)
        self.dims = dims_from_config(config, num_states)
        dev = self.device
        self.actor = NetBank("actor", self.dims, self.A, dev, with_optimizer=True)
        self.critic = NetBank("critic", self.dims, self.A, dev, with_optimizer=True)
        self.t_actor = NetBank("actor", self.dims, self.A, dev)
        self.t_critic = NetBank("critic", self.dims, self.A, dev)
        if seeds is None:
            self.S = 1
            gen = torch.Generator().manual_seed(int(getattr(config, "random_seed", 1) if seed is None else seed))
            self.actor.init_reference(gen)
            self.critic.init_reference(gen)
        else:
            self.S = len(seeds)
            if self.S < 1 or self.G % self.S:
                raise ValueError(f"{self.G} groups cannot be split into {self.S} runs")
            for s, k in enumerate(seeds):
                gen = torch.Generator().manual_seed(int(k))      # the actor, then the critic: the stand-alone draw order
                agents = self.run_agents(s)
                self.actor.init_reference(gen, agents)
                self.critic.init_reference(gen, agents)
        self.sync_targets()
        self.hp = None
        if overrides is not None:
            from .config import run_configs
            confs = run_configs(config, seeds, overrides)
            rows = [[float(c.gamma), float(c.actor_lr), float(c.critic_lr), float(c.tau)] for c in confs]
            Gr = self.G // self.S
            self.hp = torch.tensor([rows[(a % self.G) // Gr] for a in range(self.A)], dtype=torch.float32, device=dev)
        self.loss = torch.zeros(self.A, 2, dtype=torch.float32, device=dev)
        self._ws = None
        self._act_ws = None
        self.io = _lib.LearnIO()

    def run_agents(self, s: int) -> torch.Tensor:
        """Agent indices of run s, in the stand-alone run's agent order m*Gr + g' (agent m*G + s*Gr + g' here)."""
        Gr = self.G // self.S
        return (torch.arange(self.M).unsqueeze(1) * self.G + s * Gr + torch.arange(Gr).unsqueeze(0)).reshape(-1)

    def sync_targets(self):
        """target.set_weights(online.get_weights())  (trainer.py:130-131)."""
        self.t_actor.flat.copy_(self.actor.flat)
        self.t_critic.flat.copy_(self.critic.flat)

    def _workspace(self, rows):
        need = self.lib.avd_ddpg_workspace_bytes(C.byref(self.dims), self.A, rows, self.precision)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    # ------------------------------------------------------------------ acting
    def act(self, native_state: torch.Tensor, out: torch.Tensor, envs_per_group: int):
        """actor(state) for every vehicle of a BatchedPlatoons batch: native_state [4, M, P] (P = G*E),
        out [M, P] (e.g. env.action_mu).  Row n = m*P + p belongs to agent n // E."""
        d = self.dims
        M, P = native_state.shape[1], native_state.shape[2]
        if M != self.M or P != self.G * envs_per_group:
            raise ValueError("state batch does not match the population")
        rows = envs_per_group
        need = self.lib.avd_forward_workspace_bytes(C.byref(d), self.A, rows, 0, self.precision)
        if self._act_ws is None or self._act_ws.numel() < need:
            self._act_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.avd_actor_forward(C.byref(d), self.A, rows, _lib.ptr(self.actor.flat), _lib.ptr(native_state), 1,
                                              M * P, float(self.config.action_high), _lib.ptr(out), _lib.ptr(self._act_ws),
                                              self._act_ws.numel(), self.precision, _lib.current_stream()))
        return out

    # ------------------------------------------------------------------ learning
    def learn(self, s, a, r, s2, *, apply_updates: bool = True, apply_mask: Optional[torch.Tensor] = None,
              rows_per_agent: Optional[int] = None):
        """One Trainer.learn for every agent.  s, s2: [A*R, 4]; a, r: [A*R] (float32, CUDA, contiguous).
        Gradients land in self.actor.grad / self.critic.grad ([A, n_trainable], `trainable_variables` order);
        with apply_updates the weights, Adam state and targets are updated in place."""
        R = self.R if rows_per_agent is None else int(rows_per_agent)
        n = self.A * R
        for t, width in ((s, 4), (s2, 4)):
            if t.shape != (n, width) or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"state batches must be contiguous float32 [A*R={n}, 4]")
        conf, io = self.config, self.io
        ws = self._workspace(R)
        io.dims, io.A, io.apply_updates, io.rows_per_agent = self.dims, self.A, int(apply_updates), R
        io.gamma, io.action_high, io.tau = float(conf.gamma), float(conf.action_high), float(conf.tau)
        io.actor_lr, io.critic_lr = float(conf.actor_lr), float(conf.critic_lr)
        io.adam_beta1, io.adam_beta2, io.adam_eps = 0.9, 0.999, 1e-7     # tf.keras.optimizers.Adam defaults
        io.s, io.a, io.r, io.s2 = s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr()
        io.actor, io.critic = self.actor.flat.data_ptr(), self.critic.flat.data_ptr()
        io.t_actor, io.t_critic = self.t_actor.flat.data_ptr(), self.t_critic.flat.data_ptr()
        io.actor_grad, io.critic_grad = self.actor.grad.data_ptr(), self.critic.grad.data_ptr()
        io.actor_m, io.actor_v = self.actor.m.data_ptr(), self.actor.v.data_ptr()
        io.critic_m, io.critic_v = self.critic.m.data_ptr(), self.critic.v.data_ptr()
        io.actor_t, io.critic_t = self.actor.step.data_ptr(), self.critic.step.data_ptr()
        io.apply_mask = None if apply_mask is None else apply_mask.data_ptr()
        io.loss = self.loss.data_ptr()
        io.workspace, io.workspace_bytes = ws.data_ptr(), ws.numel()
        io.precision, io.s_stride = self.precision, 4         # the replay gather writes 4 state words per row; dims.ns of them are read
        io.agent_hp = None if self.hp is None else self.hp.data_ptr()
        _lib.check(self.lib.avd_ddpg_learn(C.byref(io), _lib.current_stream()))
        return self.critic.grad, self.actor.grad

    def apply_gradients(self, apply_mask: Optional[torch.Tensor] = None):
        """optimizer.apply_gradients for both nets with whatever is in .grad (trainer.py:348-349 / 420-425)."""
        self._refuse_table("apply_gradients")
        conf = self.config
        for bank, lr in ((self.critic, conf.critic_lr), (self.actor, conf.actor_lr)):
            _lib.check(self.lib.avd_adam_apply(_lib.ptr(bank.flat), bank.total, _lib.ptr(bank.grad), bank.n_train, _lib.ptr(bank.m),
                                               _lib.ptr(bank.v), _lib.ptr(bank.step), _lib.ptr(apply_mask), self.A, bank.n_train,
                                               float(lr), 0.9, 0.999, 1e-7, _lib.current_stream()))

    def apply_gradients_and_soft_update(self, apply_mask: Optional[torch.Tensor] = None):
        """apply_gradients + soft_update in three launches (Adam and Polyak of a net share one pass over its weights)."""
        conf, a, c = self.config, self.actor, self.critic
        _lib.check(self.lib.avd_adam_polyak_apply2(
            _lib.ptr(a.flat), _lib.ptr(self.t_actor.flat), a.total, _lib.ptr(a.grad), a.n_train, _lib.ptr(a.m), _lib.ptr(a.v), _lib.ptr(a.step),
            a.n_train, float(conf.actor_lr), _lib.ptr(c.flat), _lib.ptr(self.t_critic.flat), c.total, _lib.ptr(c.grad), c.n_train, _lib.ptr(c.m),
            _lib.ptr(c.v), _lib.ptr(c.step), c.n_train, float(conf.critic_lr), _lib.ptr(apply_mask), self.A, 0.9, 0.999, 1e-7, float(conf.tau),
            _lib.ptr(self.hp), _lib.current_stream()))

    def _refuse_table(self, what):
        if self.hp is not None:
            raise NotImplementedError(f"{what} applies the config's scalars; a population with per-run overrides updates through "
                                      "learn() or apply_gradients_and_soft_update()")

    def soft_update(self, apply_mask: Optional[torch.Tensor] = None):
        """ddpgagent.update_target + set_weights for every agent (trainer.py:352-356)."""
        self._refuse_table("soft_update")
        for tgt, onl in ((self.t_critic, self.critic), (self.t_actor, self.actor)):
            _lib.check(self.lib.avd_polyak_update(_lib.ptr(tgt.flat), _lib.ptr(onl.flat), _lib.ptr(apply_mask), self.A, onl.total,
                                                  float(self.config.tau), _lib.current_stream()))


class BatchedTrainer:
    """The hot loop of workers/trainer.py:251-271 for a whole population on one GPU (rank):

        actor(prev_state) -> OU noise + clip -> Platoon.step -> ReplayBuffer.add        (advance_environment, 282-302)
        if buffer_counter > batch_size: sample -> learn -> [FRL stash] -> Adam, Polyak   (train_all_models, 304-359)
        [federated round on the steps the predicates select]                             (400-456)

    G platoon-groups x E environments per group x M followers; the M*G agents' weights live in a
    DDPGPopulation, the M*G*E replay rings in ReplayRings, the platoons in BatchedPlatoons.  Everything stays
    on the device; the host only launches kernels (optionally a captured CUDA graph of the whole step).
    Per-platoon episode handling replaces the reference's "any platoon terminal ends the episode for all"
    (trainer.py:268-269): a platoon that terminates or reaches steps_per_episode is reset inside the env kernel.

    seeds=[k_0, ..., k_{S-1}] hosts S independent runs of num_groups x envs_per_group platoons each: run s behaves like the
    stand-alone trainer with random_seed = k_s (its draws, initial weights, FRL systems, episodes and reward log) and owns groups
    [s*Gr, (s+1)*Gr) of the G = S*Gr here (Gr = num_groups), so its platoons and rings are contiguous.  Single GPU only.

    overrides=[d_0, ..., d_{S-1}] (with seeds, one dict per run) makes the batch a hyperparameter sweep: run s reproduces the stand-alone
    trainer built from run_config(s), a copy of conf with random_seed = k_s and the fields of d_s set.  The keys may be actor_lr,
    critic_lr, gamma, tau, std_dev and theta (config.SWEEP_KEYS); seeds may repeat.  Two runs that share a seed write CSV files of the
    same names (reward_logs()), so give their logs different output directories.
    """

    def __init__(self, conf, num_groups: int, envs_per_group: int = 1, *, ring_capacity=None, rank: int = 0, world: int = 1,
                 process_group=None, precision: int = 0, seed=None, track_kinematics: bool = False, fed_transport: str = "auto",
                 seeds=None, overrides=None):
        from .config import run_configs
        from .environment import BatchedPlatoons, RunTable
        from .replaybuffer import ReplayRings
        # validated before anything is allocated; without seeds: the one run of conf
        if seeds is None and overrides is not None:
            raise ValueError("overrides needs seeds: one dict per run")
        self._run_confs = run_configs(conf, [int(getattr(conf, "random_seed", 1))] if seeds is None else seeds, overrides)
        self.overrides = None if overrides is None else [dict(d) for d in overrides]
        self.S = 1 if seeds is None else len(seeds)
        self.conf, self.Gr, self.E, self.M = conf, int(num_groups), int(envs_per_group), int(conf.pl_size)
        self.G = self.Gr * self.S
        self.P = self.G * self.E
        self.rank, self.world = rank, world
        self.seeds, self.runs = None, None
        if seeds is not None:
            if world > 1 or process_group is not None:
                raise ValueError("seeds: the runs of a batch live on one GPU (world must be 1)")
            if is_fed_enabled(conf) and is_model_weight_updates_enabled(conf):
                # run()'s per-run loop has gradient rounds only, so even one seed would silently train unlike its stand-alone run
                raise NotImplementedError("weights-mode FRL is not available for trainers built with seeds")
            ou = {} if overrides is None else dict(ou_sigma=[float(c.std_dev) for c in self._run_confs],
                                                   ou_theta=[float(c.theta) for c in self._run_confs])
            self.runs = RunTable(seeds, self.Gr * self.E, torch.device("cuda", torch.cuda.current_device()), **ou)
            self.seeds = self.runs.seeds
        seed = int(getattr(conf, "random_seed", 1) if seed is None else seed)
        cap = int(conf.buffer_size if ring_capacity is None else ring_capacity)
        self.rings = ReplayRings(cap, self.M, self.P, int(conf.batch_size), seed=seed, ring_id_base=rank * self.M * self.P, runs=self.runs)
        self.env = BatchedPlatoons(self.P, self.M, conf, platoon_id_base=rank * self.P, seed=seed, ring=self.rings,
                                   clock=self.rings.clock, auto_reset=True, collect_stats=True, track_kinematics=track_kinematics,
                                   reward_history=int(conf.weighted_window) if is_fed_enabled(conf) and conf.weighted_average_enabled else 0,
                                   runs=self.runs)
        self.pop = DDPGPopulation(self.G, self.M, conf, num_states=self.env.num_states, rows_per_agent=self.E * int(conf.batch_size),
                                  seed=seed, precision=precision, seeds=self.seeds, overrides=self.overrides)
        self.fed = None
        if is_fed_enabled(conf):
            from .server.federated import FederatedAggregator
            self.fed = FederatedAggregator(self.pop, conf, process_group=process_group, transport=fed_transport, runs=self.S)
        self.buffer_counter = 0          # == ReplayBuffer.buffer_counter of every ring
        self.step_in_run = 0             # bookkeeping only
        # What the FRL scheduling predicates see (workers/trainer.py:232, 251: `ep`, `i`).  run() counts real episodes and zeroes
        # the step index at every env.reset(); the free-running step() loop (per-platoon auto-reset, no global episode) uses the
        # nominal episode clock: a new episode every conf.steps_per_episode steps.
        self.episode = 0
        self.step_in_episode = 0
        self._in_run = False
        self.fed_weights = None          # [systems][members] device tensor of the current episode's FedAvg weights, or None
        self._fed_w = None
        self.graph = None
        self._dev = None                 # _DeviceEpisodes of run() on the device (trainers built with seeds)
        self.env.reset()

    @property
    def gpu_launches(self):
        """Kernels launched by libavddpg_b200 in this process so far (counted at the launch sites inside the library)."""
        return int(self.pop.lib.avd_kernel_launches())

    def step(self, learn: bool = True, host_leader_exog: Optional[torch.Tensor] = None):
        """One environment step for every platoon + one learn() for every agent (when the buffers hold more than
        batch_size transitions, trainer.py:322).  host_leader_exog: pinned host tensor [P] with the leaders'
        exogenous inputs (the reference draws them on the host, trainer.py:292-295); None = drawn on the device."""
        env, pop, rings, conf = self.env, self.pop, self.rings, self.conf
        pop.act(env.native_state, env.action_mu, self.E)
        if host_leader_exog is not None:
            env.leader_exog.copy_(host_leader_exog, non_blocking=True)
            env.step_native(explore=True, leader_exog=True, advance_clock=False)
        else:
            env.step_native(explore=True, gen_exog=True, advance_clock=False)
        rings.clock.advance(step=1, ring=1)
        self.buffer_counter += 1
        if learn and self.buffer_counter > conf.batch_size:
            s, a, r, s2 = rings.sample(advance_clock=True)
            ep, i = self.episode, self.step_in_episode
            fed_step = self.fed is not None and is_valid_update_step(conf, i)
            pop.learn(s, a, r, s2, apply_updates=not fed_step)          # trainer.py:345: local update unless FRL step
            if self.fed is not None:
                grads = is_valid_step_for_federated_training_with_gradients(conf, ep, i)
                weights = is_valid_step_for_federated_training_with_weights(conf, ep, i)
                if grads or weights:
                    w = self._frl_weights(ep)                           # trainer.py:331-333: None before the weighting window
                    if grads:
                        self.fed.aggregate_gradients(w, write_back=False)
                    if weights:
                        self.fed.aggregate_weights(w)
        self.step_in_run += 1
        self.step_in_episode += 1
        if not self._in_run and self.step_in_episode >= int(conf.steps_per_episode):
            self.step_in_episode, self.episode = 0, self.episode + 1

    def _frl_weights(self, episode: int):
        """FedAvg weights of this round, [systems][members] on the device: |1 / mean(last weighted_window episodic rewards)| per
        agent (Trainer.get_weight, trainer.py:385-398), from the ring of finished-episode rewards the env kernel keeps.  None while
        is_weighted_fed_enabled is false (plain mean)."""
        conf = self.conf
        self.fed_weights = None
        if not is_weighted_fed_enabled(conf, episode):
            return None
        if self._fed_w is None:
            self._fed_w = torch.zeros(self.fed.n_systems, self.fed.n_members, dtype=torch.float32, device=self.pop.device)
        _lib.check(self.pop.lib.avd_fed_weights_from_history(_lib.ptr(self.env.ep_hist), int(conf.weighted_window), self.M, self.G, self.E,
                                                             _lib.ptr(self._fed_w), 0 if self.fed.inter else 1, _lib.current_stream()))
        self.fed_weights = self._fed_w
        return self._fed_w

    def frl_weight_lists(self, run: Optional[int] = None):
        """(fed_weights[g][m], fed_weight_sums[g][m]) of the last federated round as nested lists of np.float32, the layout
        update_reward_list records (trainer.py:521-528), or (None, None) when the round was unweighted.  fed_weight_sums is the sum
        over ALL members of the system -- over every rank's platoons for interfrl (it travels through the exchange).
        run: only the groups of that run (trainers built with seeds)."""
        if self.fed is None or self.fed_weights is None or self.fed.last_weight_sums is None:
            return None, None
        w = self.fed_weights.cpu().numpy().astype(np.float32)            # [systems][members]
        sums = self.fed.last_weight_sums.cpu().numpy().astype(np.float32)  # [systems]
        return self._weight_lists(w, sums, run)

    def _weight_lists(self, w, sums, run):
        groups = range(self.G) if run is None else range(run * self.Gr, (run + 1) * self.Gr)
        if self.fed.inter:      # systems = (follower m, run k) = m*S + k, members = the run's groups g'
            Gr, S = self.Gr, self.S
            return ([[w[m * S + g // Gr, g % Gr] for m in range(self.M)] for g in groups],
                    [[sums[m * S + g // Gr] for m in range(self.M)] for g in groups])
        return ([[w[g, m] for m in range(self.M)] for g in groups], [[sums[g] for m in range(self.M)] for g in groups])

    def episodic_rewards(self, run: Optional[int] = None):
        """Cumulative reward of the current episode per agent, [G][M] nested lists of np.float32 (the reference's
        all_episodic_reward_counters, trainer.py:249, 321); with E environments per group: the mean over the group's platoons.
        run: only the groups of that run, [Gr][M] (trainers built with seeds)."""
        r = self.env.ep_reward.reshape(self.M, self.G, self.E).mean(dim=2).t().contiguous().cpu().numpy().astype(np.float32)
        groups = range(self.G) if run is None else range(run * self.Gr, (run + 1) * self.Gr)
        return [[r[g, m] for m in range(self.M)] for g in groups]

    def run_config(self, s: int):
        """Run s's effective configuration: a copy of conf with the run's random_seed and overrides applied."""
        if not 0 <= s < self.S:
            raise IndexError(f"run {s} outside {self.S} runs")
        return copy.copy(self._run_confs[s])

    def reward_logs(self):
        """One results.RewardLog per run, each on the run's configuration (run_config), so that generate_csvs writes its files as
        ..._seed{k_s}.csv (the files the reference's accumr aggregates).  Runs that share a seed (a sweep over overrides) produce
        files of the same names: write their logs into different directories."""
        from .results import RewardLog
        return [RewardLog(self.run_config(s), num_platoons=self.Gr, num_models=self.M) for s in range(self.S)]

    def run_weights(self, s: int, group: int = 0):
        """Run s's weights: (actors, critics) with actors[m] / critics[m] the Keras `.weights` arrays of follower m of the run's group
        `group` -- what results.save_weights writes, or what a G = 1 DDPGPopulation takes (set_weights) for evaluator.run."""
        if not 0 <= s < self.S or not 0 <= group < self.Gr:
            raise IndexError(f"run {s} / group {group} outside {self.S} runs of {self.Gr} groups")
        agents = [m * self.G + s * self.Gr + group for m in range(self.M)]
        return [self.pop.actor.get_weights(a) for a in agents], [self.pop.critic.get_weights(a) for a in agents]

    def run(self, episodes: int, reward_log=None, *, global_break: bool = True, learn: bool = True, any_terminal_group=None,
            reward_logs=None):
        """The episode loop of Trainer.run (workers/trainer.py:232-273) for the whole population: every episode resets ALL
        platoons (246-249), runs up to conf.steps_per_episode steps (251), ends early for everybody when ANY platoon reports a
        terminal state (268-269; `global_break=False` lets the other platoons finish) and appends the episodic rewards to
        `reward_log` (an avddpg_b200.results.RewardLog; trainer.py:273, 510-517).  A trainer built with seeds runs this loop per run
        on the device (see _run_device) and takes `reward_logs`, one RewardLog per run (reward_logs()).  In-kernel auto-reset is
        switched off for the duration, so episodes line up across platoons exactly like the reference's; without seeds one D2H read
        of the done flags per step is the price (the free-running `step()` loop used by the benchmark never synchronises).  `any_terminal_group`: a
        torch.distributed group over which "any platoon terminal" is agreed (one 1-word all_reduce(MAX) per step) so that platoons
        sharded over several GPUs still end their episodes together (SURVEY.md section 8e: opt-in).  Returns the number of env steps."""
        if self.runs is not None:
            if reward_log is not None or any_terminal_group is not None:
                raise ValueError("a trainer with runs takes reward_logs (one per run) and no any_terminal_group")
            return self._run_device(episodes, reward_logs, global_break, learn)
        if reward_logs is not None:
            raise ValueError("reward_logs is for trainers built with seeds; pass reward_log")
        env, conf = self.env, self.conf
        saved = env.auto_reset
        env.auto_reset = False
        self._in_run = True
        steps = 0
        try:
            for _ in range(int(episodes)):
                env.reset()
                self.step_in_episode = 0                       # trainer.py:251: `i` restarts with every episode
                for _ in range(int(conf.steps_per_episode)):
                    self.step(learn=learn)
                    steps += 1
                    if global_break:
                        term = (env.done & 1).any()
                        if any_terminal_group is not None:
                            import torch.distributed as dist
                            term = term.to(torch.int32)
                            dist.all_reduce(term, op=dist.ReduceOp.MAX, group=any_terminal_group)
                        if bool(term.item()):
                            break
                if reward_log is not None:
                    fw, fws = self.frl_weight_lists() if is_weighted_fed_enabled(conf, self.episode) else (None, None)
                    reward_log.update_reward_list(self.episodic_rewards(), fw, fws)
                if self.fed is not None:
                    self.fed.check_health()                        # a peer that missed a round's barrier is an error, not a hang
                self.episode += 1
        finally:
            env.auto_reset = saved
            self._in_run = False
        return steps

    def _run_runs(self, episodes: int, reward_logs, global_break: bool, learn: bool):
        """The host reference of _run_device (one D2H read of the done flags and host-built masks per step).  run() for S runs: each run keeps its own episode index and step-in-episode counter, ends its episode when one of ITS
        platoons is terminal (global_break) or after steps_per_episode steps, then logs its rewards and resets only its own
        platoons.  FRL predicates and the weighting window are evaluated per run.  A run that has finished its episodes is frozen
        (its agents take no further update) while the others go on, so its weights end where the stand-alone run's do."""
        env, conf, S = self.env, self.conf, self.S
        if reward_logs is not None and len(reward_logs) != S:
            raise ValueError(f"{len(reward_logs)} reward logs for {S} runs")
        spe, Pr = int(conf.steps_per_episode), self.Gr * self.E
        saved = env.auto_reset
        env.auto_reset = False
        self._in_run = True
        self._run_ep, self._run_i = [self.episode] * S, [0] * S
        left = [int(episodes)] * S
        self.run_episode_steps = [[] for _ in range(S)]     # [run][episode]: env steps of each episode of this call
        steps = 0
        try:
            if any(left):
                env.reset()
            while any(left):
                active = [n > 0 for n in left]
                self._step_runs(learn, active)
                steps += 1
                term = (env._done & 1).view(S, Pr).any(dim=1).tolist() if global_break else [False] * S
                ending = []
                for k in range(S):
                    if active[k]:
                        self._run_i[k] += 1
                        if term[k] or self._run_i[k] >= spe:
                            ending.append(k)
                for k in ending:
                    if reward_logs is not None:
                        fw, fws = self.frl_weight_lists(k) if is_weighted_fed_enabled(conf, self._run_ep[k]) else (None, None)
                        reward_logs[k].update_reward_list(self.episodic_rewards(k), fw, fws)
                    self.run_episode_steps[k].append(self._run_i[k])
                    self._run_ep[k] += 1
                    self._run_i[k] = 0
                    left[k] -= 1
                restart = [k for k in ending if left[k] > 0]
                if restart:
                    env.reset(self._run_mask(restart, per="platoon"))
            self.episode += int(episodes)
        finally:
            env.auto_reset = saved
            self._in_run = False
        return steps

    def _run_mask(self, runs, per: str = "agent") -> torch.Tensor:
        """uint8 device mask over agents [A] (a = m*G + k*Gr + g') or platoons [P] (p = k*Pr + p') of the listed runs."""
        f = torch.zeros(self.S, dtype=torch.uint8)
        f[list(runs)] = 1
        if per == "platoon":
            m = f.repeat_interleave(self.Gr * self.E)
        else:
            m = f.view(1, self.S, 1).expand(self.M, self.S, self.Gr).reshape(-1)
        return m.to(self.pop.device)

    def _step_runs(self, learn: bool, active):
        """step() with per-run FRL predicates (run k at episode _run_ep[k], step _run_i[k]); runs not in `active` are frozen.  Runs on
        an FRL step skip the local update (trainer.py:345) and take the federated round if it is a gradients round; the others take
        their local Adam / Polyak step through the learn call's apply mask."""
        env, pop, rings, conf, S = self.env, self.pop, self.rings, self.conf, self.S
        pop.act(env.native_state, env.action_mu, self.E)
        env.step_native(explore=True, gen_exog=True, advance_clock=False)
        rings.clock.advance(step=1, ring=1)
        self.buffer_counter += 1
        if learn and self.buffer_counter > conf.batch_size:
            s, a, r, s2 = rings.sample(advance_clock=True)
            fed_step = [active[k] and self.fed is not None and is_valid_update_step(conf, self._run_i[k]) for k in range(S)]
            grads = [fed_step[k] and is_valid_step_for_federated_training_with_gradients(conf, self._run_ep[k], self._run_i[k])
                     for k in range(S)]
            local = [k for k in range(S) if active[k] and not fed_step[k]]
            pop.learn(s, a, r, s2, apply_updates=bool(local), apply_mask=self._run_mask(local))
            if any(grads):
                mask = self._run_mask([k for k in range(S) if grads[k]])
                if self.fed.apply_mask is not None:
                    mask = mask & self.fed.apply_mask
                self.fed.aggregate_gradients(self._frl_weights_runs(), write_back=False, apply_mask=mask)
        self.step_in_run += 1

    def _frl_weights_runs(self):
        """_frl_weights with per-run weighting windows: the FedAvg weights of every run past its window, 1 for the others (a plain
        mean).  None while no run is past its window."""
        conf = self.conf
        plain = [k for k in range(self.S) if not is_weighted_fed_enabled(conf, self._run_ep[k])]
        if len(plain) == self.S:
            return None
        w = self._frl_weights(self._run_ep[[k for k in range(self.S) if k not in plain][0]])
        for k in plain:
            if self.fed.inter:      # [M*S][Gr]: system m*S + k
                w.view(self.M, self.S, self.Gr)[:, k, :] = 1.0
            else:                   # [G][M]: systems k*Gr .. (k+1)*Gr - 1
                w.view(self.S, self.Gr, self.M)[k] = 1.0
        return w

    # ------------------------------------------------------------------ the per-run episode loop on the device
    RUN_LOG_SLOTS = 64          # episode records per run one graph launch of _run_device can log before the host drains them

    def _run_device(self, episodes: int, reward_logs, global_break: bool, learn: bool):
        """_run_runs with the loop on the device, bit-identical to it: after every step the episode controller (avd_episode_control)
        ends episodes, logs them and writes the next step's masks, and a conditional CUDA graph repeats the step while runs have
        episodes left.  Each graph launch runs until every run is done, a run's log is full (run_log_slots records) or, without
        learning yet, the rings reach batch_size transitions; then the host synchronises once, drains the log into the reward logs
        and, if needed, launches again.  The graphs (with and without learning, per starting state buffer) are built on first use
        by capturing the same library calls _step_runs makes, and cached."""
        env, conf, S = self.env, self.conf, self.S
        if reward_logs is not None and len(reward_logs) != S:
            raise ValueError(f"{len(reward_logs)} reward logs for {S} runs")
        episodes = int(episodes)
        self._run_ep, self._run_i = [self.episode] * S, [0] * S
        self.run_episode_steps = [[] for _ in range(S)]
        if episodes <= 0:
            self.episode += episodes
            return 0
        L = self._device_episodes()
        bs, lib = int(conf.batch_size), self.pop.lib
        saved = env.auto_reset
        env.auto_reset = False
        self._in_run = True
        steps = rounds = 0
        try:
            env.reset()
            flags = (_lib.EPISODE_HAVE_WEIGHTS if self.fed_weights is not None else 0) | \
                    (_lib.EPISODE_HAVE_SUMS if self.fed is not None and self.fed.last_weight_sums is not None else 0)
            L.ctr.copy_(torch.tensor([[episodes] * S, [self.episode] * S, [0] * S, [0] * S], dtype=torch.int32))
            L.state.copy_(torch.tensor([self.buffer_counter, 0, 0, 0, flags], dtype=torch.int64))
            while True:
                learning = learn and self.buffer_counter >= bs
                L.state[3].fill_(bs if learn and not learning else _NEVER)
                g = self._loop_graph(learning, global_break)
                _lib.check(lib.avd_loop_graph_launch(g, _lib.current_stream()))
                st, ctr = L.state.tolist(), L.ctr.tolist()          # the one synchronisation per launch
                taken = st[1] - steps
                steps, rounds = st[1], st[2]
                self.buffer_counter = st[0]
                self.step_in_run += taken
                env._cur ^= taken & 1
                self._drain_episode_log(ctr[3], reward_logs)
                if not any(n > 0 for n in ctr[0]):
                    break
                if taken == 0 and not any(ctr[3]):
                    raise RuntimeError("device episode loop made no progress")
                L.ctr[3].zero_()
            self._run_ep, self._run_i = ctr[1], ctr[2]
            self.episode += episodes
            if self.fed is not None:
                self.fed.rounds += rounds
                if st[4] & _lib.EPISODE_HAVE_SUMS:
                    self.fed.last_weight_sums = self.fed.wsum
                if st[4] & _lib.EPISODE_HAVE_WEIGHTS:
                    self.fed_weights = self._fed_w
        finally:
            env.auto_reset = saved
            self._in_run = False
        return steps

    def _drain_episode_log(self, nrec, reward_logs):
        """The records of one launch, in each run's order: run_episode_steps and reward_logs[k].update_reward_list with the same values
        _run_runs passes (episodic_rewards' expression on the logged ep_reward rows, frl_weight_lists' layout)."""
        L, M, G, E, Gr = self._dev, self.M, self.G, self.E, self.Gr
        J = max(nrec)
        if J == 0:
            return
        lens, wrec = L.log_len[:J].tolist(), L.log_weighted[:J].tolist()
        if reward_logs is not None:
            n = M * self.P
            rew = torch.stack([L.log_reward[j, :n].reshape(M, G, E).mean(dim=2).t().contiguous() for j in range(J)])
            rew = rew.cpu().numpy().astype(np.float32)
            if L.log_w is not None:
                w, ws = L.log_w[:J].cpu().numpy().astype(np.float32), L.log_wsum[:J].cpu().numpy().astype(np.float32)
        for k in range(self.S):
            for j in range(nrec[k]):
                self.run_episode_steps[k].append(lens[j][k])
                if reward_logs is not None:
                    fw, fws = self._weight_lists(w[j], ws[j], k) if wrec[j][k] else (None, None)
                    reward_logs[k].update_reward_list([[rew[j, g, m] for m in range(M)] for g in range(k * Gr, (k + 1) * Gr)], fw, fws)

    def _device_episodes(self):
        slots = max(1, int(self.RUN_LOG_SLOTS))
        if self._dev is None or self._dev.slots != slots:
            self._free_loop_graphs()
            self._dev = _DeviceEpisodes(self, slots)
        return self._dev

    def _episode_control(self, mode, learning=False, cont_handles=(), step_handles=(None, None)):
        """One avd_episode_control launch; step_handles: the (round, local) IF handles of the next step, or None each."""
        io = _lib.EpisodeIO.from_buffer_copy(self._dev.io)
        io.mode, io.learn, io.n_cont_handles = mode, int(learning), len(cont_handles)
        for j, h in enumerate(cont_handles):
            io.cont_handle[j] = h
        (rh, lh) = step_handles
        io.has_round_handle, io.round_handle = int(rh is not None), rh or 0
        io.has_local_handle, io.local_handle = int(lh is not None), lh or 0
        _lib.check(self.pop.lib.avd_episode_control(C.byref(io), _lib.current_stream()))

    def _loop_graph(self, learning: bool, global_break: bool):
        """The cached loop graph for the current state buffer:
            ARM -> WHILE (continue) { step A -> controller -> reset(mask)
                                      IF (continue) { step B -> controller -> reset(mask) } }
        with a learning step = act -> env step -> sample -> learn (gradients) -> IF (local) {Adam / Polyak} -> IF (round) {FRL round}.
        Step B reads the buffer step A writes, so every iteration ends on the buffer it started from; a launch that ends after step A
        leaves the other buffer current, and the next launch takes the graph built for that one."""
        L, env, lib = self._dev, self.env, self.pop.lib
        L.io.global_break = int(global_break)
        key = (learning, global_break, env._cur)
        if key in L.graphs:
            return L.graphs[key]
        rounds = learning and L.rounds
        self._warm_loop(learning)
        n = 2 + (2 if learning else 0) + (2 if rounds else 0)
        hs = (C.c_uint64 * 6)()
        g = C.c_void_p()
        _lib.check(lib.avd_loop_graph_create(C.byref(g), n, hs))
        h_while, h_b = int(hs[0]), int(hs[1])
        la, lb = (int(hs[2]), int(hs[3])) if learning else (None, None)
        ra, rb = (int(hs[4]), int(hs[5])) if rounds else (None, None)
        st = L.streams
        fed = self.fed
        saved = (self.buffer_counter, self.step_in_run, env._cur, env._launches,
                 None if fed is None else (fed.rounds, fed.last_weight_sums))

        def body():
            self._device_step(g, learning, (ra, la), st[2])
            self._episode_control(_lib.EPISODE_STEP, learning, (h_while, h_b), (rb, lb))
            env.reset(L.reset_mask)

            def step_b():
                self._device_step(g, learning, (rb, lb), st[3])
                self._episode_control(_lib.EPISODE_STEP, learning, (h_while,), (ra, la))
                env.reset(L.reset_mask)
            self._graph_cond(g, h_b, 0, st[2], step_b)

        try:
            _lib.check(lib.avd_loop_graph_capture_begin(g, st[0].cuda_stream))
            with torch.cuda.stream(st[0]):
                self._episode_control(_lib.EPISODE_ARM, learning, (h_while,), (ra, la))
                self._graph_cond(g, h_while, 1, st[1], body)
            _lib.check(lib.avd_loop_graph_capture_end(g, st[0].cuda_stream))
        except BaseException:
            lib.avd_loop_graph_destroy(g)
            raise
        finally:      # capturing executes nothing on the device
            self.buffer_counter, self.step_in_run, env._cur, env._launches = saved[:4]
            if fed is not None:
                fed.rounds, fed.last_weight_sums = saved[4]
        L.graphs[key] = g
        return g

    def _graph_cond(self, g, handle, kind, child, body):
        """body()'s launches, enqueued on the current stream's position, inside an IF (kind 0) / WHILE (1) node on `handle`."""
        lib = self.pop.lib
        _lib.check(lib.avd_loop_graph_cond_begin(g, handle, kind, torch.cuda.current_stream().cuda_stream, child.cuda_stream))
        with torch.cuda.stream(child):
            body()
        _lib.check(lib.avd_loop_graph_cond_end(g, child.cuda_stream))

    def _device_step(self, g, learning: bool, handles, child):
        """_step_runs with its masks read from the device (the controller wrote them): the local Adam / Polyak step (the same launch
        learn() makes with apply_updates) and the FRL round each behind an IF node, so a step without them costs nothing for them."""
        env, pop, rings, L = self.env, self.pop, self.rings, self._dev
        pop.act(env.native_state, env.action_mu, self.E)
        env.step_native(explore=True, gen_exog=True, advance_clock=False)
        rings.clock.advance(step=1, ring=1)
        self.buffer_counter += 1
        if learning:
            s, a, r, s2 = rings.sample(advance_clock=True)
            pop.learn(s, a, r, s2, apply_updates=False)
            round_handle, local_handle = handles
            self._graph_cond(g, local_handle, 0, child, lambda: pop.apply_gradients_and_soft_update(L.learn_mask))
            if L.rounds:
                self._graph_cond(g, round_handle, 0, child, self._device_round)
        self.step_in_run += 1

    def _device_round(self):
        """The gradients round of _step_runs on the device masks: with weighting, _frl_weights_runs' weights (the runs before their
        window take 1, which avd_fed_reduce2 sums exactly like its NULL weights)."""
        L, conf, env = self._dev, self.conf, self.env
        w = None
        if L.round_w is not None:
            _lib.check(self.pop.lib.avd_fed_weights_from_history(_lib.ptr(env.ep_hist), int(conf.weighted_window), self.M, self.G, self.E,
                                                                 _lib.ptr(L.round_w), 0 if self.fed.inter else 1, _lib.current_stream()))
            self._episode_control(_lib.EPISODE_WEIGHTS)
            w = L.round_w
        self.fed.aggregate_gradients(w, write_back=False, apply_mask=L.round_mask)

    def _warm_loop(self, learning: bool):
        """Allocate everything a captured step uses (nothing may allocate during capture) and create the learn step's side stream."""
        pop, rings = self.pop, self.rings
        pop.act(self.env.native_state, self.env.action_mu, self.E)     # the first step overwrites action_mu
        if learning:
            rings._alloc_sample_buffers()
            pop.learn(rings.s, rings.a, rings.r, rings.s2, apply_updates=False)     # gradients and losses: every learn step rewrites them
            if self.fed is not None:
                self.fed._buffer(pop.actor.n_train, pop.critic.n_train)

    def _free_loop_graphs(self):
        if self._dev is not None:
            for g in self._dev.graphs.values():
                self.pop.lib.avd_loop_graph_destroy(g)
            self._dev.graphs.clear()

    def __del__(self):
        try:
            self._free_loop_graphs()
        except Exception:       # noqa: BLE001 -- interpreter shutdown: the library may already be gone
            pass

    def capture(self, warmup: int = 3):
        """Capture one full step (learn included) into a CUDA graph; afterwards `replay()` costs one launch.  The host-side FRL
        schedule is frozen into the graph, so capture is refused unless every step takes the same branch (fed_update_delay_steps == 1
        and every episode a federated one); the cross-GPU exchange keeps its epoch / buffer half in device memory
        (FederatedAggregator), so replays synchronise exactly like eager rounds."""
        assert self.buffer_counter > self.conf.batch_size, "fill the buffers past batch_size before capturing"
        if self.fed is not None:
            conf = self.conf
            uniform = (int(conf.fed_update_delay_steps) == 1 and int(conf.fed_update_count) == 1 and float(conf.fed_cutoff_ratio) >= 1.0
                       and not (conf.weighted_average_enabled and self.episode < int(conf.weighted_window)))
            if not uniform:
                raise RuntimeError("capture() needs a step-invariant FRL schedule: fed_update_delay_steps == 1, fed_update_count == 1, "
                                   "fed_cutoff_ratio >= 1 and, with weighted averaging, an episode past the weighting window")
            if not self.fed.graph_safe:
                raise RuntimeError(f"the {self.fed.transport} FRL transport cannot be captured into a CUDA graph")
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                self.step()
        torch.cuda.current_stream().wait_stream(stream)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        cur, counters = self.env._cur, (self.buffer_counter, self.step_in_run, self.step_in_episode, self.episode)
        n0 = self.pop.lib.avd_kernel_launches()
        with torch.cuda.graph(self.graph):
            self.step()
            self.step()      # two steps per graph so the ping-pong state buffers end where they started
        self.kernels_per_step = (self.pop.lib.avd_kernel_launches() - n0) // 2
        assert self.env._cur == cur
        self.buffer_counter, self.step_in_run, self.step_in_episode, self.episode = counters     # capturing executes nothing on the device
        return self.graph

    def replay(self):
        self.graph.replay()
        self.buffer_counter += 2
        self.step_in_run += 2
        self.step_in_episode += 2
        spe = int(self.conf.steps_per_episode)
        if not self._in_run and self.step_in_episode >= spe:
            self.step_in_episode, self.episode = self.step_in_episode - spe, self.episode + 1


_NEVER = (1 << 63) - 1      # avd_episode_state.learn_from when no prefix stop applies


class _DeviceEpisodes:
    """Device state of BatchedTrainer._run_device: the episode controller's counters, masks and log (avd_episode_io) and the
    cached loop graphs."""

    def __init__(self, tr: "BatchedTrainer", slots: int):
        dev, conf, fed = tr.pop.device, tr.conf, tr.fed
        S, P, A, M = tr.S, tr.P, tr.pop.A, tr.M
        u8, i32, f32 = (dict(dtype=t, device=dev) for t in (torch.uint8, torch.int32, torch.float32))
        self.slots = slots
        self.state = torch.zeros(5, dtype=torch.int64, device=dev)            # avd_episode_state (flags in the low half of word 4)
        self.ctr = torch.zeros(4, S, **i32)                                    # left, ep, i, nrec
        self.reset_mask, self.learn_mask = torch.zeros(P, **u8), torch.zeros(A, **u8)
        self.round_mask = None if fed is None else torch.zeros(A, **u8)
        self.rounds = fed is not None and is_fed_enabled(conf) and bool(conf.fed_enabled) and is_gradient_updates_enabled(conf)
        weighted = fed is not None and bool(conf.weighted_average_enabled)
        if weighted and tr._fed_w is None:
            tr._fed_w = torch.zeros(fed.n_systems, fed.n_members, **f32)
        self.round_w = torch.zeros(fed.n_systems, fed.n_members, **f32) if weighted else None
        pitch = (M * P + 127) // 128 * 128      # every record starts 512-byte aligned, like env.ep_reward (same reduction in mean())
        self.log_reward = torch.zeros(slots, pitch, **f32)
        self.log_w = torch.zeros(slots, fed.n_systems, fed.n_members, **f32) if weighted else None
        self.log_wsum = torch.zeros(slots, fed.n_systems, **f32) if weighted else None
        self.log_len, self.log_weighted = torch.zeros(slots, S, **i32), torch.zeros(slots, S, **i32)
        self.streams = [torch.cuda.Stream() for _ in range(4)]                # capture: top level, loop body, step B / round, round in B
        self.graphs = {}
        io = self.io = _lib.EpisodeIO()
        io.runs, io.platoons_per_run, io.groups_per_run, io.M = S, tr.Gr * tr.E, tr.Gr, M
        io.steps_per_episode, io.global_break = int(conf.steps_per_episode), 1
        io.fed = 0 if fed is None else (1 if fed.inter else 2)
        io.fed_gradients = int(self.rounds)
        if fed is not None:
            io.fed_update_delay_steps, io.fed_update_count = int(conf.fed_update_delay_steps), int(conf.fed_update_count)
            io.fed_cutoff_episode = max(-(1 << 31), min(int(conf.fed_cutoff_episode), (1 << 31) - 1))
        io.weighted, io.weighted_window = int(bool(conf.weighted_average_enabled)), int(conf.weighted_window)
        io.log_slots = slots
        io.state = self.state.data_ptr()
        io.left, io.ep, io.i, io.nrec = (self.ctr[j].data_ptr() for j in range(4))
        io.done, io.ep_reward = tr.env._done.data_ptr(), tr.env.ep_reward.data_ptr()
        io.reset_mask, io.learn_mask = self.reset_mask.data_ptr(), self.learn_mask.data_ptr()
        ptr = lambda t: None if t is None else t.data_ptr()
        io.round_mask, io.fed_apply_mask = ptr(self.round_mask), ptr(None if fed is None else fed.apply_mask)
        io.fed_w, io.round_w, io.wsum = ptr(tr._fed_w if weighted else None), ptr(self.round_w), ptr(None if fed is None else fed.wsum)
        io.log_reward, io.log_w, io.log_wsum = self.log_reward.data_ptr(), ptr(self.log_w), ptr(self.log_wsum)
        io.log_len, io.log_weighted, io.log_pitch = self.log_len.data_ptr(), self.log_weighted.data_ptr(), pitch


class HostStepPipeline:
    """Drives `BatchedTrainer.step()` from HOST buffers without ever draining the GPU.

    The reference's loop is host-driven: the leaders' exogenous inputs are drawn on the host every step
    (workers/trainer.py:292-295) and the rewards / losses are read there (trainer.py:321, 496-504).  A synchronous version of
    that hand-off costs one GPU idle period per step (result read -> next input -> first launch).  Here both directions are
    double-buffered in pinned memory: step k copies its inputs from buffer k & 1 and its results (reward / done statistics of
    `env.stats`, critic and actor losses) into result buffer k & 1, and `submit()` returns the results of step k - 1 while step
    k runs.  Every step's inputs go host -> device and every step's results come back; the host merely reads them one step late.

        pipe = HostStepPipeline(trainer)
        for k in range(n):
            pipe.input_buffer().normal_(0, 0.1)      # leaders' exogenous inputs of step k, [P] pinned
            prev = pipe.submit()                     # None for k = 0, else pinned [M + 1 + 2 A] of step k - 1
        last = pipe.drain()
    """

    def __init__(self, trainer: "BatchedTrainer"):
        self.tr = trainer
        env, pop = trainer.env, trainer.pop
        assert env.stats is not None, "construct the environment with collect_stats=True"
        self.n_stats = int(env.stats.numel())
        self.h_in = [torch.zeros(env.P, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.h_out = [torch.zeros(self.n_stats + int(pop.loss.numel()), dtype=torch.float32).pin_memory() for _ in range(2)]
        self.done = [torch.cuda.Event(), torch.cuda.Event()]
        self.k = 0

    @property
    def h2d_bytes_per_step(self) -> int:
        return int(self.h_in[0].numel()) * 4

    @property
    def d2h_bytes_per_step(self) -> int:
        return int(self.h_out[0].numel()) * 4

    def input_buffer(self) -> torch.Tensor:
        """Pinned [P] buffer to fill with the next step's leader inputs; its previous use (two steps ago) has completed."""
        return self.h_in[self.k & 1]

    def submit(self, learn: bool = True) -> Optional[torch.Tensor]:
        tr, b = self.tr, self.k & 1
        tr.env.stats.zero_()
        tr.step(learn=learn, host_leader_exog=self.h_in[b])
        self.h_out[b][: self.n_stats].copy_(tr.env.stats, non_blocking=True)
        self.h_out[b][self.n_stats:].copy_(tr.pop.loss.reshape(-1), non_blocking=True)
        self.done[b].record()
        self.k += 1
        if self.k < 2:
            return None
        self.done[b ^ 1].synchronize()               # step k - 1: finished while step k was being enqueued
        return self.h_out[b ^ 1]

    def drain(self) -> Optional[torch.Tensor]:
        """Results of the last submitted step."""
        if self.k == 0:
            return None
        b = (self.k - 1) & 1
        self.done[b].synchronize()
        return self.h_out[b]


class Trainer:
    """Reference-shaped wrapper: ``learn`` on single-agent model objects (trainer.py:472-508)."""

    def __init__(self, base_dir=None, timestamp=None, debug_enabled=False, conf=None):
        self.base_dir, self.timestamp, self.debug_enabled, self.conf = base_dir, timestamp, debug_enabled, conf
        self._ws = None

    def learn(self, rbuffer, actor_model, critic_model, target_actor, target_critic, indices=None):
        """-> (critic_grad, actor_grad): lists of tensors ordered like ``trainable_variables``."""
        lib = _lib.load()
        conf = self.conf
        s, a, r, s2 = rbuffer.sample(indices)
        d = critic_model.bank.dims
        n = s.shape[0]

        def pad4(x):
            if x.shape[1] == 4:
                return x.contiguous()
            out = torch.zeros(n, 4, dtype=torch.float32, device=x.device)
            out[:, : x.shape[1]] = x
            return out

        s, s2 = pad4(s), pad4(s2)                   # 3-state Model A batches travel in 4-word rows (s_stride = 4, dims.ns = 3)
        a, r = a.reshape(-1).contiguous(), r.reshape(-1).contiguous()
        dev = s.device
        ag = torch.zeros(1, actor_model.bank.n_train, dtype=torch.float32, device=dev)
        cg = torch.zeros(1, critic_model.bank.n_train, dtype=torch.float32, device=dev)
        need = lib.avd_ddpg_workspace_bytes(C.byref(d), 1, n, 0)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        io = _lib.LearnIO()
        io.dims, io.A, io.apply_updates, io.rows_per_agent = d, 1, 0, n
        io.gamma, io.action_high = float(conf.gamma), float(conf.action_high)
        io.s, io.a, io.r, io.s2 = s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr()
        io.actor, io.critic = actor_model.bank.flat.data_ptr(), critic_model.bank.flat.data_ptr()
        io.t_actor, io.t_critic = target_actor.bank.flat.data_ptr(), target_critic.bank.flat.data_ptr()
        io.actor_grad, io.critic_grad = ag.data_ptr(), cg.data_ptr()
        io.workspace, io.workspace_bytes = self._ws.data_ptr(), self._ws.numel()
        io.s_stride = 4
        _lib.check(lib.avd_ddpg_learn(C.byref(io), _lib.current_stream()))
        critic_grad = [critic_model.bank.view(nm, 0, cg) for nm in critic_model.bank.trainable_names]
        actor_grad = [actor_model.bank.view(nm, 0, ag) for nm in actor_model.bank.trainable_names]
        return critic_grad, actor_grad


# ---- FRL scheduling predicates (workers/trainer.py:631-695), pure host logic ---------------------------
def is_fed_enabled(conf) -> bool:
    return (conf.fed_method == conf.interfrl or conf.fed_method == conf.intrafrl) and (conf.framework == conf.dcntrl)


def is_gradient_updates_enabled(conf) -> bool:
    return conf.aggregation_method == conf.gradients


def is_model_weight_updates_enabled(conf) -> bool:
    return conf.aggregation_method == conf.weights


def is_weighted_fed_enabled(conf, training_episode: int) -> bool:
    return bool(conf.weighted_average_enabled and training_episode >= conf.weighted_window)


def is_valid_update_episode(conf, training_episode: int) -> bool:
    return bool(conf.fed_enabled and (training_episode % conf.fed_update_count) == 0 and training_episode <= conf.fed_cutoff_episode)


def is_valid_update_step(conf, training_step: int) -> bool:
    return (training_step % conf.fed_update_delay_steps) == 0


def is_valid_step_for_federated_training_with_gradients(conf, training_episode, training_step):
    return (is_fed_enabled(conf) and is_valid_update_episode(conf, training_episode) and is_valid_update_step(conf, training_step)
            and is_gradient_updates_enabled(conf))


def is_valid_step_for_federated_training_with_weights(conf, training_episode, training_step):
    return (is_fed_enabled(conf) and is_valid_update_episode(conf, training_episode) and is_valid_update_step(conf, training_step)
            and is_model_weight_updates_enabled(conf))
