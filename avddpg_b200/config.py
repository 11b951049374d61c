"""Hot-path configuration: the attribute names of the reference's ``Config`` (src/config.py:14-219)
that the environment / agent / trainer path actually reads (SURVEY.md §8a), with the same defaults.

Any object carrying these attributes works wherever a ``conf`` is expected -- including a reference
``Config`` instance or the ``SimpleNamespace`` its ``conf.json`` loader returns (src/util.py:33-35) -- so
the classes in this package are drop-ins for workers/trainer.py.  Reporting/plotting/file-name fields
of the reference Config are out of scope and not reproduced.
"""
from __future__ import annotations

import copy
import ctypes as C
import math

from . import _lib

# value tables rather than a wall of assignments; citations are src/config.py line numbers
_CONSTANTS = dict(modelA="ModelA", modelB="ModelB", dcntrl="decentralized", cntrl="centralized",
                  interfrl="interfrl", intrafrl="intrafrl", nofrl="normal", weights="weights",
                  gradients="gradients", exact="exact", euler="euler", normal="normal", uniform="uniform")

_DEFAULTS = dict(
    # federated learning (25-37)
    fed_method="normal", framework="decentralized", weighted_average_enabled=True, weighted_window=10,
    fed_update_count=1, fed_cutoff_ratio=1.0, fed_update_delay=0.1, aggregation_method="gradients",
    intra_directional_averaging=False,
    # environment (39-72)
    num_platoons=1, pl_size=2, pl_leader_reset_a=0, reset_max_u=0.100, pl_leader_tau=0.1, method="euler",
    model="ModelB", timegap=1.0, dyn_coeff=0.1, reward_ep_coeff=0.4, reward_ev_coeff=0.2, reward_u_coeff=0.2,
    reward_jerk_coeff=0.2, max_ep=20, max_ev=20, reset_ep_max=1.5, reset_max_ev=1.5, reset_max_a=0.05,
    reset_ep_eval_max=1, reset_ev_eval_max=1, reset_a_eval_max=0.03, action_high=2.5, action_low=-2.5,
    re_scalar=1, terminal_reward=0.5,
    # trainer (75-107)
    can_terminate=True, random_seed=1, evaluation_seed=6, rand_gen="normal", rand_states=True,
    total_time_steps=1000000, sample_rate=0.1, episode_sim_time=60, gamma=0.99, centrl_hidd_mult=1.2,
    reward_averaging_window=40, critic_lr=0.0005, actor_lr=0.00005, std_dev=0.02, theta=0.15, ou_dt=1e-2,
    tau=0.001, batch_size=64, buffer_size=100000, show_env=False,
    # models (112-117)
    actor_layer1_size=256, actor_layer2_size=128, critic_layer1_size=256, critic_act_layer_size=48,
    critic_layer2_size=128,
)


class Config:
    """Attribute bag with the reference's names and defaults; keyword overrides are applied before the
    derived fields are computed (the reference computes them once in its constructor, config.py:88-94)."""

    def __init__(self, **overrides):
        for k, v in {**_CONSTANTS, **_DEFAULTS}.items():
            setattr(self, k, v)
        unknown = set(overrides) - set(_DEFAULTS)
        if unknown:
            raise AttributeError(f"unknown Config fields: {sorted(unknown)}")
        for k, v in overrides.items():
            setattr(self, k, v)
        self.refresh_derived()

    def refresh_derived(self):
        self.steps_per_episode = int(self.episode_sim_time / self.sample_rate)            # config.py:88
        self.fed_update_delay_steps = int(self.fed_update_delay / self.sample_rate)       # config.py:89
        self.number_of_episodes = int(self.total_time_steps / self.steps_per_episode)     # config.py:91
        self.fed_cutoff_episode = int(self.fed_cutoff_ratio * self.number_of_episodes)    # config.py:94
        self.fed_enabled = (self.fed_method in (self.interfrl, self.intrafrl)) and self.framework == self.dcntrl


def _get(conf, name):
    return getattr(conf, name) if hasattr(conf, name) else _DEFAULTS[name]


def env_params_from_config(conf, M: int, rand_states: bool = True, evaluator_states_enabled: bool = False,
                           steps_per_episode=None) -> _lib.EnvParams:
    """Fill the C struct the kernels read.  Reset-mode selection follows Vehicle.reset
    (src/environment.py:534-555)."""
    if not (1 <= M <= _lib.AVD_MAX_FOLLOWERS):
        raise ValueError(f"Platoon of length {M}: supported range is 1..{_lib.AVD_MAX_FOLLOWERS}")
    model = _get(conf, "model")
    if model not in ("ModelA", "ModelB"):
        raise ValueError(f"unknown vehicle model {model!r}")   # the reference falls into UnboundLocalError here
    method = _get(conf, "method")
    if method not in ("euler", "exact"):
        raise ValueError(f"unknown discretisation {method!r}")
    rand_gen = _get(conf, "rand_gen")
    if rand_gen not in ("normal", "uniform"):
        raise ValueError(f"unknown rand_gen {rand_gen!r}")
    p = _lib.EnvParams()
    p.M = M
    p.num_states = 3 if model == "ModelA" else 4
    p.model_a = int(model == "ModelA")
    p.can_terminate = int(bool(_get(conf, "can_terminate")))
    p.centralized = int(_get(conf, "framework") == "centralized")
    p.rand_uniform = int(rand_gen == "uniform")
    if evaluator_states_enabled:
        p.reset_mode = 1
        if rand_states:
            trio = (_get(conf, "reset_ep_eval_max"), _get(conf, "reset_ev_eval_max"), _get(conf, "reset_a_eval_max"))
        else:
            trio = (_get(conf, "reset_ep_max"), _get(conf, "reset_max_ev"), _get(conf, "reset_max_a"))
    else:
        p.reset_mode = 0 if rand_states else 1
        trio = (_get(conf, "reset_ep_max"), _get(conf, "reset_max_ev"), _get(conf, "reset_max_a"))
    p.reset_ep, p.reset_ev, p.reset_a = (float(v) for v in trio)
    spe = steps_per_episode
    if spe is None:
        spe = getattr(conf, "steps_per_episode", int(_get(conf, "episode_sim_time") / _get(conf, "sample_rate")))
    p.steps_per_episode = int(spe)
    p.max_ep, p.max_ev = float(_get(conf, "max_ep")), float(_get(conf, "max_ev"))
    p.action_high, p.action_low = float(_get(conf, "action_high")), float(_get(conf, "action_low"))
    p.rew_ep, p.rew_ev = float(_get(conf, "reward_ep_coeff")), float(_get(conf, "reward_ev_coeff"))
    p.rew_u, p.rew_jerk = float(_get(conf, "reward_u_coeff")), float(_get(conf, "reward_jerk_coeff"))
    p.re_scalar, p.terminal_reward = float(_get(conf, "re_scalar")), float(_get(conf, "terminal_reward"))
    p.reset_leader_a, p.reset_u = float(_get(conf, "pl_leader_reset_a")), float(_get(conf, "reset_max_u"))
    p.ou_theta, p.ou_dt = float(_get(conf, "theta")), float(_get(conf, "ou_dt"))
    p.ou_sigma, p.ou_mean = float(_get(conf, "std_dev")), 0.0
    _lib.check(_lib.load().avd_env_build_matrices(C.byref(p), int(method == "exact"), float(_get(conf, "sample_rate")),
                                                  float(_get(conf, "timegap")), float(_get(conf, "dyn_coeff")),
                                                  float(_get(conf, "pl_leader_tau"))))
    return p


# Config fields a run of a batched sweep may override (BatchedTrainer(..., seeds=..., overrides=...)): the scalars the learn step
# and the OU noise read.  Every other field would change shapes or the environment and is shared by all runs of a batch.
SWEEP_KEYS = ("actor_lr", "critic_lr", "gamma", "tau", "std_dev", "theta")


def run_configs(conf, seeds, overrides=None) -> list:
    """Effective configuration of every run of a batch: a copy of `conf` with random_seed = seeds[s] and the fields of overrides[s]
    set.  overrides: None, or one dict per seed whose keys are among SWEEP_KEYS and whose values are finite numbers; a missing key
    keeps conf's value.  Raises ValueError for any other key, a non-finite or non-numeric value, or a length mismatch.  Host only."""
    if overrides is not None:
        if seeds is None:
            raise ValueError("overrides needs seeds: one dict per run")
        overrides = list(overrides)
        if len(overrides) != len(seeds):
            raise ValueError(f"{len(overrides)} overrides for {len(seeds)} seeds")
    out = []
    for s, k in enumerate(seeds):
        c = copy.copy(conf)
        c.random_seed = k
        d = {} if overrides is None else overrides[s]
        if not isinstance(d, dict):
            raise ValueError(f"overrides[{s}] must be a dict, got {type(d).__name__}")
        bad = sorted(set(d) - set(SWEEP_KEYS))
        if bad:
            raise ValueError(f"overrides[{s}]: {bad} cannot differ between the runs of a batch (allowed: {', '.join(SWEEP_KEYS)})")
        for key, v in d.items():
            try:
                f = float(v)
            except (TypeError, ValueError):
                raise ValueError(f"overrides[{s}][{key!r}] = {v!r} is not a number") from None
            if isinstance(v, bool) or not math.isfinite(f):
                raise ValueError(f"overrides[{s}][{key!r}] = {v!r} is not a finite number")
            setattr(c, key, f)
        out.append(c)
    return out
