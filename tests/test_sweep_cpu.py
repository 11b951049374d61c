"""Host-only checks of a hyperparameter sweep's configuration (config.run_configs, BatchedTrainer(..., seeds, overrides)): which
fields a run may override, and what is refused before anything touches a device."""
import math

import pytest

from avddpg_b200.config import SWEEP_KEYS, Config, run_configs


def test_run_configs_apply_overrides_on_copies():
    conf = Config(pl_size=3, gamma=0.99, actor_lr=5e-5)
    over = [{}, {"actor_lr": 1e-3, "gamma": 0.5}, {"std_dev": 0.1, "theta": 0.3, "tau": 0.05, "critic_lr": 2e-3}]
    confs = run_configs(conf, [4, 4, 9], over)
    assert [c.random_seed for c in confs] == [4, 4, 9]
    assert (confs[0].actor_lr, confs[0].gamma) == (5e-5, 0.99)
    assert (confs[1].actor_lr, confs[1].gamma, confs[1].critic_lr) == (1e-3, 0.5, conf.critic_lr)
    assert (confs[2].std_dev, confs[2].theta, confs[2].tau, confs[2].critic_lr) == (0.1, 0.3, 0.05, 2e-3)
    assert all(c.pl_size == 3 and c is not conf for c in confs)
    assert (conf.random_seed, conf.actor_lr, conf.gamma) == (1, 5e-5, 0.99), "the base configuration is left alone"
    assert set(SWEEP_KEYS) == {"actor_lr", "critic_lr", "gamma", "tau", "std_dev", "theta"}


@pytest.mark.parametrize("seeds,overrides", [
    ([1, 2], [{"batch_size": 32}, {}]),                 # changes shapes
    ([1, 2], [{}, {"pl_size": 4}]),
    ([1], [{"gamma": math.nan}]),
    ([1], [{"tau": math.inf}]),
    ([1], [{"actor_lr": -math.inf}]),
    ([1], [{"std_dev": "0.1x"}]),
    ([1], [{"theta": True}]),
    ([1, 2], [{}]),                                     # length mismatch
    ([1], [{}, {}]),
    (None, [{}]),                                       # overrides need seeds
    ([1], [[("gamma", 0.5)]]),
])
def test_run_configs_refusals(seeds, overrides):
    with pytest.raises(ValueError):
        run_configs(Config(), seeds, overrides)


@pytest.mark.parametrize("kw", [dict(seeds=[1, 2], overrides=[{"batch_size": 32}, {}]), dict(seeds=[1, 2], overrides=[{}]),
                                dict(overrides=[{"gamma": 0.5}]), dict(seeds=[3], overrides=[{"gamma": math.nan}])])
def test_trainer_refuses_bad_overrides_before_touching_a_device(kw):
    from avddpg_b200.trainer import BatchedTrainer
    with pytest.raises(ValueError):
        BatchedTrainer(Config(pl_size=2, batch_size=16, buffer_size=64), 1, 1, ring_capacity=64, **kw)
