"""run() of a trainer built with seeds runs its per-run episode loop on the device (episode controller + conditional CUDA graph).  Two
identical trainers, one through run() and one through the host reference loop (_run_runs), must agree.

Without learning everything is compared bit for bit.  With learning the learn step's float atomics make weights reproducible to
rounding only, even between two identical trainers, so floats are held to the bars of test_gpu_runs.py while every integer (episode
lengths, step and round counts, Adam step counters, episode counters, clock, host counters) must still match exactly."""
import numpy as np
import pytest
import torch

from test_gpu_runs import BARS

pytestmark = pytest.mark.gpu

SEEDS = [4, 9, 21]


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _conf(**over):
    from avddpg_b200.config import Config
    base = dict(pl_size=2, batch_size=16, buffer_size=256, can_terminate=True, reset_ep_max=0.5, reset_max_ev=0.5, max_ep=1.0, max_ev=1.0,
                episode_sim_time=3.0, fed_method="normal", reward_averaging_window=2)
    base.update(over)
    return Config(**base)


def _np(t):
    return t.detach().cpu().numpy()


def _twins(conf, Gr, E, seeds, precision=0, overrides=None):
    from avddpg_b200.trainer import BatchedTrainer
    mk = lambda: BatchedTrainer(conf, Gr, E, seeds=seeds, ring_capacity=256, precision=precision, overrides=overrides)
    return mk(), mk()


def _margins(tr, conf):
    margins, orig = [], tr._step_runs

    def step(*a, **kw):
        orig(*a, **kw)
        x = tr.env.state.abs()
        margins.append(min(float((x[..., 0] - conf.max_ep).abs().min()), float((x[..., 1] - conf.max_ev).abs().min())))
    tr._step_runs = step
    return margins


def _run_both(dev, host, episodes, learn, calls=1):
    ld, lh = dev.reward_logs(), host.reward_logs()
    margins = _margins(host, host.conf)
    for _ in range(calls):
        nd = dev.run(episodes, reward_logs=ld, learn=learn)
        nh = host._run_runs(episodes, lh, True, learn)
        assert nd == nh, (nd, nh)
        assert dev.run_episode_steps == host.run_episode_steps
    if learn:    # DESIGN.md section 4: a state this close to a threshold could flip a break on a last-bit difference
        assert min(margins) > 1e-4, f"a state came within {min(margins):.1e} of a terminal threshold"
    return ld, lh


def _close(got, want, tol, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, what
    if want.size:
        err = np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-3))
        assert err < tol, (what, err)


def _compare(dev, host, ld, lh, exact, precision=0):
    for a in ("buffer_counter", "step_in_run", "episode", "_run_ep", "_run_i"):
        assert getattr(dev, a) == getattr(host, a), a
    assert dev.env._cur == host.env._cur
    for name in ("episode", "step_in_episode", "_done"):
        assert torch.equal(getattr(dev.env, name), getattr(host.env, name)), name
    assert torch.equal(dev.rings.clock.t, host.rings.clock.t)
    for b in ("actor", "critic"):
        assert torch.equal(getattr(dev.pop, b).step, getattr(host.pop, b).step), b
    if dev.fed is not None:
        assert dev.fed.rounds == host.fed.rounds
        assert (dev.fed_weights is None) == (host.fed_weights is None)
        assert (dev.fed.last_weight_sums is None) == (host.fed.last_weight_sums is None)
    floats = [("ep_reward", dev.env.ep_reward, host.env.ep_reward), ("state", dev.env._x, host.env._x),
              ("ou", dev.env.ou_state, host.env.ou_state)]
    written = min(dev.buffer_counter, dev.rings.capacity)          # the rest of the ring is uninitialised memory
    floats.append(("rings", dev.rings.data[:written], host.rings.data[:written]))
    if dev.env.ep_hist is not None:
        floats.append(("ep_hist", dev.env.ep_hist, host.env.ep_hist))
    for b in ("actor", "critic", "t_actor", "t_critic"):
        floats.append((b, getattr(dev.pop, b).flat, getattr(host.pop, b).flat))
    for b in ("actor", "critic"):
        floats += [(b + ".m", getattr(dev.pop, b).m, getattr(host.pop, b).m), (b + ".v", getattr(dev.pop, b).v, getattr(host.pop, b).v)]
    if dev.fed_weights is not None:
        floats += [("fed_w", dev.fed_weights, host.fed_weights), ("wsum", dev.fed.last_weight_sums, host.fed.last_weight_sums)]
    for k in range(dev.S):
        for f in ("all_ep_reward_lists", "all_avg_reward_lists", "all_fed_weights", "all_fed_weight_sums"):
            g, w = getattr(ld[k], f), getattr(lh[k], f)
            if exact:
                assert np.array_equal(np.asarray(g, dtype=np.float64), np.asarray(w, dtype=np.float64)), (k, f)
                assert [[type(x) for x in r] for r in g] == [[type(x) for x in r] for r in w], (k, f)
            else:
                _close(g, w, BARS[precision][1], (k, f))
    for name, g, w in floats:
        if exact:
            assert torch.equal(g, w), name
        else:
            _close(_np(g), _np(w), BARS[precision][2], name)


@pytest.mark.parametrize("learn", [False, True])
def test_run_loop_per_run_breaks(learn):
    """(a) no FRL, runs ending their episodes at different steps, E = 2."""
    _need_gpu()
    dev, host = _twins(_conf(), 1, 2, SEEDS)
    ld, lh = _run_both(dev, host, 4, learn)
    assert len({tuple(x) for x in dev.run_episode_steps}) > 1, "runs should break at different steps"
    _compare(dev, host, ld, lh, exact=not learn)
    if learn:
        assert int(dev.pop.actor.step.max()) > 0


@pytest.mark.parametrize("precision", [0, 2])
def test_run_loop_weighted_interfrl(precision):
    """(b) weighted interfrl every second step with a one-episode window: on one step some runs take a round, some a local update,
    and some use plain means while others are past their window."""
    _need_gpu()
    conf = _conf(fed_method="interfrl", weighted_average_enabled=True, weighted_window=1, fed_update_delay=0.2)
    assert conf.fed_update_delay_steps == 2
    dev, host = _twins(conf, 2, 1, SEEDS, precision=precision)
    ld, lh = _run_both(dev, host, 4, True)
    assert dev.fed.rounds > 0 and dev.fed_weights is not None
    assert all(len(log.all_fed_weights[0][0]) > 0 for log in ld)
    _compare(dev, host, ld, lh, exact=False, precision=precision)


def test_run_loop_intrafrl_directional():
    """(c) intrafrl with directional averaging (follower 0 never takes the round)."""
    _need_gpu()
    conf = _conf(pl_size=3, fed_method="intrafrl", intra_directional_averaging=True, weighted_average_enabled=False)
    dev, host = _twins(conf, 2, 1, SEEDS)
    assert dev.fed.apply_mask is not None
    ld, lh = _run_both(dev, host, 3, True)
    assert dev.fed.rounds > 0
    _compare(dev, host, ld, lh, exact=False)


def test_run_loop_overrides_same_seed():
    """(d) a sweep with two runs of one seed."""
    _need_gpu()
    dev, host = _twins(_conf(), 1, 1, [5, 5, 8], overrides=[dict(std_dev=0.03), dict(std_dev=0.2, tau=0.002), dict(gamma=0.9)])
    ld, lh = _run_both(dev, host, 3, False)
    _compare(dev, host, ld, lh, exact=True)
    ld, lh = _run_both(dev, host, 2, True)
    _compare(dev, host, ld, lh, exact=False)


def test_run_loop_prefix_then_learning():
    """(e) a first call that starts with empty rings (the prefix graph without learning hands over to the learning graph), then a
    second call on the other state buffer parity."""
    _need_gpu()
    conf = _conf(batch_size=32, fed_method="interfrl", weighted_average_enabled=True, weighted_window=2)
    dev, host = _twins(conf, 2, 1, SEEDS)
    ld, lh = _run_both(dev, host, 2, True, calls=2)
    assert dev.buffer_counter > conf.batch_size
    _compare(dev, host, ld, lh, exact=False)


def test_run_loop_small_log_budget():
    """(f) a log budget of one record per run: the call drains the log and relaunches many times; without learning all is bitwise."""
    _need_gpu()
    dev, host = _twins(_conf(fed_method="interfrl", weighted_average_enabled=True, weighted_window=1), 2, 1, SEEDS)
    dev.RUN_LOG_SLOTS = 1
    launches = []
    orig = dev._drain_episode_log
    dev._drain_episode_log = lambda nrec, logs: (launches.append(1), orig(nrec, logs))
    ld, lh = _run_both(dev, host, 5, False)
    assert len(launches) >= 5
    _compare(dev, host, ld, lh, exact=True)


def test_run_loop_no_per_step_host_work():
    """Once its graphs exist, run() launches the same number of times (from the host) for 2 and for 8 episodes."""
    _need_gpu()
    dev, _ = _twins(_conf(fed_method="interfrl", weighted_average_enabled=False), 2, 1, SEEDS)
    dev.run(2)                      # builds the prefix and learning graphs
    for _ in range(20):             # until the learning graph exists for both starting state buffers
        if {(True, True, 0), (True, True, 1)} <= set(dev._dev.graphs):
            break
        dev.run(1)
    n0 = dev.gpu_launches
    s2 = dev.run(2)
    n2 = dev.gpu_launches - n0
    n0 = dev.gpu_launches
    s8 = dev.run(8)
    n8 = dev.gpu_launches - n0
    assert s8 > 3 * s2 > 0
    assert n2 == n8 <= 3, (n2, n8)
