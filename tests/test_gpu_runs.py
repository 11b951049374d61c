"""Independently seeded runs batched into one trainer (BatchedTrainer(..., seeds=[...])): run s of the batch must reproduce the
stand-alone trainer with random_seed = seeds[s].

Without learning that holds bit for bit (the run table only re-keys the Philox streams, and the actor forward is bit-identical per
row whatever the agent slot).  With learning the learn step's float atomics make weights reproducible to rounding only, so the
closed loops are held to the bars of test_gpu_loop.py (DESIGN.md section 4).
"""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SEEDS5 = [1, 2, 7, 123, (1 << 40) + 3]
BARS = {0: (2e-5, 1e-4, 5e-3), 2: (5e-4, 1e-2, 5e-2)}      # states, losses, weight updates


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _conf(**over):
    from avddpg_b200.config import Config
    return Config(**over)


def _with_seed(conf, k):
    c = copy.copy(conf)
    c.random_seed = k
    return c


def _pair(conf, Gr, E, seeds, **kw):
    from avddpg_b200.trainer import BatchedTrainer
    batched = BatchedTrainer(conf, Gr, E, seeds=seeds, **kw)
    alone = [BatchedTrainer(_with_seed(conf, k), Gr, E, **kw) for k in seeds]
    return batched, alone


def _np(t):
    return t.detach().cpu().numpy()


def test_runs_bit_exact_without_learning():
    """Observations, rewards, done flags, OU states, applied actions, ring contents, sampled indices, the finished-episode reward
    history and the episode counters of every run, bitwise, over 200 free-running steps with terminations and auto-resets."""
    _need_gpu()
    Gr, E, M = 2, 1, 3
    conf = _conf(pl_size=M, batch_size=16, buffer_size=64, can_terminate=True, max_ep=2.5, max_ev=2.5, episode_sim_time=3.0,
                 fed_method="interfrl", weighted_average_enabled=True, weighted_window=3)
    tr, alone = _pair(conf, Gr, E, SEEDS5, ring_capacity=64)
    Pr = Gr * E
    for step in range(200):
        tr.step(learn=False)
        for k, st in enumerate(alone):
            st.step(learn=False)
            sl = slice(k * Pr, (k + 1) * Pr)
            for name, got, want in (("obs", tr.env.obs[sl], st.env.obs), ("reward", tr.env.reward[sl], st.env.reward),
                                    ("done", tr.env._done[sl], st.env._done), ("ou", tr.env.ou_state[:, sl], st.env.ou_state),
                                    ("action", tr.env.action_out[:, sl], st.env.action_out)):
                assert np.array_equal(_np(got), _np(want)), (step, k, name)
    idx = _np(tr.rings.sample_indices()).reshape(M, len(SEEDS5) * Pr, -1)
    episodes = _np(tr.env.episode)
    for k, st in enumerate(alone):
        sl = slice(k * Pr, (k + 1) * Pr)
        assert np.array_equal(_np(tr.rings.data[:, :, sl]), _np(st.rings.data)), k
        assert np.array_equal(idx[:, sl], _np(st.rings.sample_indices()).reshape(M, Pr, -1)), k
        assert np.array_equal(_np(tr.env.ep_hist[:, :, sl]), _np(st.env.ep_hist)), k
        assert np.array_equal(episodes[sl], _np(st.env.episode)), k
    assert len(set(episodes.tolist())) > 1, "platoons should have reset at different steps"


def test_runs_initial_weights():
    _need_gpu()
    conf = _conf(pl_size=3, batch_size=16, buffer_size=64)
    tr, alone = _pair(conf, 2, 1, SEEDS5, ring_capacity=64)
    for k, st in enumerate(alone):
        agents = tr.pop.run_agents(k).to(tr.pop.device)
        for name in ("actor", "critic", "t_actor", "t_critic"):
            got, want = getattr(tr.pop, name).flat[agents], getattr(st.pop, name).flat
            assert torch.equal(got, want), (k, name)
    assert not torch.equal(tr.pop.actor.flat[tr.pop.run_agents(0)], tr.pop.actor.flat[tr.pop.run_agents(1)])


def _rel_update(got, want, w0):
    upd = np.linalg.norm(want - w0)
    if upd < 1e-5 * max(np.linalg.norm(w0), 1e-30):
        return 0.0 if np.linalg.norm(got - want) <= 5e-6 * np.linalg.norm(w0) else np.inf
    return float(np.linalg.norm(got - want) / upd)


FED = {
    None: dict(fed_method="normal"),
    "interfrl-weighted": dict(fed_method="interfrl", weighted_average_enabled=True, weighted_window=1),
    "intrafrl-directional": dict(fed_method="intrafrl", weighted_average_enabled=False, intra_directional_averaging=True),
}


@pytest.mark.parametrize("precision", [0, 2])
@pytest.mark.parametrize("fed", list(FED))
def test_runs_closed_loop_with_learning(precision, fed):
    """50 steps of the full training step; every run against its stand-alone trainer."""
    _need_gpu()
    Gr, E, M, seeds = 2, 2, 2, [3, 5, 11]
    conf = _conf(pl_size=M, batch_size=16, buffer_size=64, can_terminate=False, episode_sim_time=1.0, **FED[fed])
    tr, alone = _pair(conf, Gr, E, seeds, ring_capacity=64, precision=precision)
    st_tol, loss_tol, upd_tol = BARS[precision]
    banks = ("actor", "critic", "t_actor", "t_critic")
    w0 = {b: _np(getattr(tr.pop, b).flat).astype(np.float64) for b in banks}
    Pr = Gr * E
    worst_state = worst_loss = worst_upd = 0.0
    for step in range(50):
        tr.step()
        for k, st in enumerate(alone):
            st.step()
            got, want = _np(tr.env.obs[k * Pr:(k + 1) * Pr]).astype(np.float64), _np(st.env.obs).astype(np.float64)
            worst_state = max(worst_state, float(np.max(np.abs(got - want)) / np.max(np.abs(want))))
            if tr.buffer_counter > conf.batch_size:
                lg = _np(tr.pop.loss[tr.pop.run_agents(k)]).astype(np.float64)
                lw = _np(st.pop.loss).astype(np.float64)
                worst_loss = max(worst_loss, float(np.max(np.abs(lg - lw) / np.maximum(np.abs(lw), 1e-3))))
    for k, st in enumerate(alone):
        agents = tr.pop.run_agents(k)
        assert torch.equal(tr.pop.actor.step[agents.to(tr.pop.device)], st.pop.actor.step), k
        for b in banks:
            got = _np(getattr(tr.pop, b).flat[agents.to(tr.pop.device)]).astype(np.float64)
            want = _np(getattr(st.pop, b).flat).astype(np.float64)
            init = w0[b][agents.numpy()]
            bank = getattr(st.pop, b)
            for name in bank.weight_names:
                off, shape = bank.offsets[name]
                n = int(np.prod(shape))
                for a in range(got.shape[0]):
                    worst_upd = max(worst_upd, _rel_update(got[a, off:off + n], want[a, off:off + n], init[a, off:off + n]))
    print(f"runs closed loop precision={precision} fed={fed}: states {worst_state:.1e} losses {worst_loss:.1e} weight updates {worst_upd:.1e}")
    assert worst_state < st_tol, worst_state
    assert worst_loss < loss_tol, worst_loss
    assert worst_upd < upd_tol, worst_upd


def _margin_recorder(tr, conf):
    """Wrap tr.step so that after every step the smallest distance of any |e_p| / |e_v| to its terminal threshold is recorded."""
    margins, orig = [], tr.step

    def step(*a, **kw):
        orig(*a, **kw)
        x = tr.env.state.abs()
        margins.append(min(float((x[..., 0] - conf.max_ep).abs().min()), float((x[..., 1] - conf.max_ev).abs().min())))
    tr.step = step
    return margins


def _check_run_loop(conf, Gr, E, seeds, episodes, learn, tmp_path):
    """run() of a batch of runs against run() of each stand-alone trainer: episode lengths, reward logs (bitwise without learning,
    within the precision-0 bars with it), FedAvg weights recorded in the logs, Adam step counts and final weights."""
    tr, alone = _pair(conf, Gr, E, seeds, ring_capacity=256, precision=0)
    w0 = {b: _np(getattr(tr.pop, b).flat).astype(np.float64) for b in ("actor", "critic")}
    logs = tr.reward_logs()
    tr.run(episodes, reward_logs=logs, learn=learn)
    _, loss_tol, upd_tol = BARS[0]
    for k, st in enumerate(alone):
        margins = _margin_recorder(st, conf)
        log = st.reward_logs()[0]
        lengths = [st.run(1, log, learn=learn) for _ in range(episodes)]
        if learn:    # DESIGN.md section 4: a state this close to a threshold could flip a break on a last-bit difference
            assert min(margins) > 1e-4, f"seed {seeds[k]}: a state came within {min(margins):.1e} of a terminal threshold"
        assert tr.run_episode_steps[k] == lengths, (k, tr.run_episode_steps[k], lengths)
        if learn:
            for got, want in ((logs[k].all_ep_reward_lists, log.all_ep_reward_lists), (logs[k].all_fed_weights, log.all_fed_weights),
                              (logs[k].all_fed_weight_sums, log.all_fed_weight_sums)):
                got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
                assert got.shape == want.shape, k
                if want.size:
                    assert np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-3)) < loss_tol, k
            agents = tr.pop.run_agents(k).to(tr.pop.device)
            assert int(st.pop.actor.step[0]) > 0, "learning must be active"
            assert torch.equal(tr.pop.actor.step[agents], st.pop.actor.step), k
            for b in ("actor", "critic"):
                got, want = _np(getattr(tr.pop, b).flat[agents]), _np(getattr(st.pop, b).flat)
                for a in range(got.shape[0]):
                    assert _rel_update(got[a].astype(np.float64), want[a].astype(np.float64), w0[b][agents[a].item()]) < upd_tol, (k, b, a)
        else:
            assert logs[k].all_ep_reward_lists == log.all_ep_reward_lists, k
            assert logs[k].all_avg_reward_lists == log.all_avg_reward_lists, k
        out = tmp_path / f"run{k}"
        out.mkdir()
        names = logs[k].generate_csvs(str(out))
        assert names and all(f"seed{seeds[k]}" in p for p in names), names
    assert len({tuple(x) for x in tr.run_episode_steps}) > 1, "runs should break at different steps"
    return tr, logs


@pytest.mark.parametrize("learn", [False, True])
def test_runs_episode_loop_per_run_break(learn, tmp_path):
    """run(): every run ends its episodes on its own terminal platoons, logs its own rewards and resets only its own platoons."""
    _need_gpu()
    M = 2
    conf = _conf(pl_size=M, batch_size=16, buffer_size=256, can_terminate=True, reset_ep_max=0.5, reset_max_ev=0.5, max_ep=1.0,
                 max_ev=1.0, episode_sim_time=3.0, fed_method="normal", reward_averaging_window=2)
    tr, _ = _check_run_loop(conf, 1, 2, [4, 9, 21], 4, learn, tmp_path)
    actors, critics = tr.run_weights(1)
    assert len(actors) == M and len(actors[0]) == len(tr.pop.actor.weight_names) and len(critics[0]) == len(tr.pop.critic.weight_names)


def test_runs_episode_loop_per_run_frl(tmp_path):
    """run() with weighted interfrl every second step (fed_update_delay_steps = 2): every run evaluates the FRL predicates and its
    weighting window on its own episode and step counters while the runs break at different steps, so on a given step some runs
    take a federated round, some a local update, and some use plain means while others are past their window."""
    _need_gpu()
    conf = _conf(pl_size=2, batch_size=16, buffer_size=256, can_terminate=True, reset_ep_max=0.5, reset_max_ev=0.5, max_ep=1.0,
                 max_ev=1.0, episode_sim_time=3.0, fed_method="interfrl", weighted_average_enabled=True, weighted_window=1,
                 fed_update_delay=0.2, reward_averaging_window=2)
    assert conf.fed_update_delay_steps == 2
    tr, logs = _check_run_loop(conf, 2, 1, [4, 9, 21], 4, True, tmp_path)
    assert tr.fed.rounds > 0
    assert all(len(log.all_fed_weights[0][0]) > 0 for log in logs), "every run should have logged FedAvg weights past its window"


def _capture_without_learning(tr):
    """capture() records learn=True steps; the same two-step graph of learn=False steps, after one warm-up step."""
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        tr.step(learn=False)
    torch.cuda.current_stream().wait_stream(stream)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        tr.step(learn=False)
        tr.step(learn=False)
    return graph


@pytest.mark.parametrize("learn", [False, True])
def test_runs_graph_capture(learn):
    """A captured 4-run trainer: 10 replays (20 steps) against 20 eager steps of a second trainer with the same seeds."""
    _need_gpu()
    from avddpg_b200.trainer import BatchedTrainer
    seeds = [5, 6, 77, 1 << 33]
    conf = _conf(pl_size=2, batch_size=16, buffer_size=64, can_terminate=True, max_ep=2.5, max_ev=2.5, episode_sim_time=2.0,
                 fed_method="interfrl", weighted_average_enabled=False)
    kw = dict(ring_capacity=64, precision=2, seeds=seeds)
    a, b = BatchedTrainer(conf, 2, 2, **kw), BatchedTrainer(conf, 2, 2, **kw)
    for tr in (a, b):
        for _ in range(20):
            tr.step(learn=learn)
    graph = a.capture(warmup=1) if learn else _capture_without_learning(a)     # one eager warm-up step, then recording only
    b.step(learn=learn)
    for _ in range(10):
        graph.replay()
        b.step(learn=learn)
        b.step(learn=learn)
    torch.cuda.synchronize()
    assert torch.equal(a.env.episode, b.env.episode)
    if not learn:
        written = min(a.rings.clock.read()["ring_count"], a.rings.capacity)      # slots past it were never written
        for name, x, y in (("obs", a.env.obs, b.env.obs), ("ring", a.rings.data[:written], b.rings.data[:written]), ("ou", a.env.ou_state, b.env.ou_state),
                           ("actions", a.env.action_out, b.env.action_out), ("ep_reward", a.env.ep_reward, b.env.ep_reward)):
            assert torch.equal(x, y), name
        return
    st_tol, loss_tol, upd_tol = BARS[2]
    x, y = _np(a.env.obs).astype(np.float64), _np(b.env.obs).astype(np.float64)
    assert np.max(np.abs(x - y)) / np.max(np.abs(y)) < st_tol
    written = min(a.rings.clock.read()["ring_count"], a.rings.capacity)
    x, y = _np(a.rings.data[:written]).astype(np.float64), _np(b.rings.data[:written]).astype(np.float64)
    assert np.max(np.abs(x - y)) / np.max(np.abs(y)) < st_tol
    la, lb = _np(a.pop.loss).astype(np.float64), _np(b.pop.loss).astype(np.float64)
    assert np.max(np.abs(la - lb) / np.maximum(np.abs(lb), 1e-3)) < loss_tol
    assert torch.equal(a.pop.actor.step, b.pop.actor.step)


def test_runs_refusals():
    _need_gpu()
    from avddpg_b200.trainer import BatchedTrainer
    conf = _conf(pl_size=2, batch_size=16, buffer_size=64, fed_method="interfrl", aggregation_method="weights")
    for seeds in ([1, 2], [7]):          # a single run too: run() has no weights rounds, so it would silently train differently
        with pytest.raises(NotImplementedError):
            BatchedTrainer(conf, 2, 1, ring_capacity=64, seeds=seeds)
    ok = _conf(pl_size=2, batch_size=16, buffer_size=64)
    with pytest.raises(ValueError):
        BatchedTrainer(ok, 1, 1, ring_capacity=64, seeds=[1, 2], world=2)
    for bad in ([1, -1], [1 << 64]):
        with pytest.raises(ValueError):
            BatchedTrainer(ok, 1, 1, ring_capacity=64, seeds=bad)
