"""Hyperparameter sweeps as one batch (BatchedTrainer(..., seeds=[...], overrides=[...])): run s must reproduce the stand-alone
trainer built from its configuration (tr.run_config(s): random_seed = seeds[s] plus overrides[s]).

The learn step reads gamma, the learning rates and tau from a per-agent table (avd_learn_io.agent_hp), the fused FRL consumer the
learning rates and tau, and the env step the per-run OU sigma and theta (avd_runs.ou_sigma / ou_theta).  Without learning a run is
bit-identical to its stand-alone trainer; with learning the closed loops are held to the bars of test_gpu_runs.py.
"""
import numpy as np
import pytest
import torch

from oracle import ddpg_np as D
from test_gpu_runs import BARS, FED, _margin_recorder, _rel_update

pytestmark = pytest.mark.gpu

# far-apart values: gamma, learning rates 10x apart, tau
HP3 = [dict(gamma=0.5, actor_lr=1e-4, critic_lr=5e-4, tau=1e-3),
       dict(gamma=0.9, actor_lr=1e-3, critic_lr=5e-3, tau=0.05),
       dict(gamma=0.99, actor_lr=1e-2, critic_lr=5e-2, tau=0.5)]
UPD_BAR = 1e-2      # Adam / Polyak step against the oracle's step on the same gradients: relative to the step, per tensor


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _conf(**over):
    from avddpg_b200.config import Config
    return Config(**over)


def _sweep(conf, Gr, E, seeds, overrides, **kw):
    from avddpg_b200.trainer import BatchedTrainer
    tr = BatchedTrainer(conf, Gr, E, seeds=seeds, overrides=overrides, **kw)
    return tr, [BatchedTrainer(tr.run_config(k), Gr, E, **kw) for k in range(len(seeds))]


def _np(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------------------------------ 1. without learning, bit for bit
def test_sweep_bit_exact_without_learning():
    """200 free-running steps with terminations and auto-resets; runs 1 and 3 share a seed and differ in std_dev and theta."""
    _need_gpu()
    Gr, E, M = 2, 1, 3
    seeds = [1, 7, 123, 7, 2]
    over = [{}, dict(std_dev=0.05, theta=0.3), dict(gamma=0.5, actor_lr=1e-3), dict(std_dev=0.01, theta=0.05), dict(theta=0.6, tau=0.1)]
    conf = _conf(pl_size=M, batch_size=16, buffer_size=64, can_terminate=True, max_ep=2.5, max_ev=2.5, episode_sim_time=3.0,
                 fed_method="interfrl", weighted_average_enabled=True, weighted_window=3)
    tr, alone = _sweep(conf, Gr, E, seeds, over, ring_capacity=64)
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
    idx = _np(tr.rings.sample_indices()).reshape(M, len(seeds) * Pr, -1)
    episodes = _np(tr.env.episode)
    for k, st in enumerate(alone):
        sl = slice(k * Pr, (k + 1) * Pr)
        assert np.array_equal(_np(tr.rings.data[:, :, sl]), _np(st.rings.data)), k
        assert np.array_equal(idx[:, sl], _np(st.rings.sample_indices()).reshape(M, Pr, -1)), k
        assert np.array_equal(_np(tr.env.ep_hist[:, :, sl]), _np(st.env.ep_hist)), k
        assert np.array_equal(episodes[sl], _np(st.env.episode)), k
    assert len(set(episodes.tolist())) > 1, "platoons should have reset at different steps"
    a, b = slice(1 * Pr, 2 * Pr), slice(3 * Pr, 4 * Pr)        # same seed, different sigma / theta
    assert not torch.equal(tr.env.ou_state[:, a], tr.env.ou_state[:, b])
    assert not torch.equal(tr.env.obs[a], tr.env.obs[b])


# ------------------------------------------------------------------------------------------ 2. learn step against the oracle
def _nets(seed):
    rng = np.random.default_rng(seed)
    nets = [D.init_actor(rng), D.init_critic(rng), D.init_actor(rng), D.init_critic(rng)]
    for p in (nets[0], nets[2]):
        D.randomize_bn(p, rng, [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
    for p in (nets[1], nets[3]):
        D.randomize_bn(p, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")])
    for p in nets:
        for k in p:
            if k.startswith("b") and not k.startswith("be"):
                p[k] = rng.normal(0, 0.05, p[k].shape).astype(np.float32)
    nets[0]["W3"] *= 50; nets[1]["W3"] *= 300; nets[2]["W3"] *= 50; nets[3]["W3"] *= 300
    return nets


def _batch(seed, R):
    rng = np.random.default_rng(seed)
    s = rng.normal(0, 2, (R, 4)).astype(np.float32); a = rng.uniform(-2.5, 2.5, (R, 1)).astype(np.float32)
    r = -rng.uniform(0, 0.5, (R, 1)).astype(np.float32); s2 = (s + rng.normal(0, 0.2, (R, 4))).astype(np.float32)
    return s, a, r, s2


def _grad_score(precision, got, want, ab, floor):
    """Error of one gradient tensor over the bar of DESIGN.md section 4 for this precision (<= 1 passes)."""
    err = float(np.linalg.norm(got - want))
    if precision in (0, 3):
        return float(np.max(np.abs(got - want)) / max(np.max(np.abs(want)), 1e-12)) / 2e-4
    if precision == 1:      # >= 1000 rows: rel-L2 2e-2, max 4e-2, against a quarter of the net's gradient norm for cancelling tensors
        e2 = err / max(float(np.linalg.norm(want)), floor)
        em = float(np.max(np.abs(got - want))) / max(float(np.max(np.abs(want))), floor / np.sqrt(got.size))
        return max(e2 / 2e-2, em / 4e-2)
    return max(err / max(float(np.linalg.norm(ab)), 1e-300) / 8e-3, err / max(float(np.linalg.norm(want)), 1e-300) / 2e-2)


LOSS_BAR = {0: 1e-4, 1: 1e-3, 2: 2e-4, 3: 1e-4}


def _learn_score(precision, pop, i, net4, batch, gamma, worst_of=None):
    """max over agent i's gradient tensors and losses of error / bar against oracle.learn with this gamma (worst_of: a list that
    receives the (score, what) of every tensor and loss)."""
    ocg, oag, info = D.learn(*net4, batch, gamma=gamma, high=2.5, with_abs=True)
    worst = 0.0
    items = [] if worst_of is None else worst_of
    for bank, ref, ab in ((pop.critic, ocg, info["critic_abs"]), (pop.actor, oag, info["actor_abs"])):
        floor = 0.25 * float(np.sqrt(sum(np.sum(np.square(ref[n].astype(np.float64))) for n in bank.trainable_names)))
        for name in bank.trainable_names:
            got = bank.view(name, i, bank.grad).cpu().numpy().astype(np.float64)
            want = ref[name].reshape(got.shape).astype(np.float64)
            items.append((_grad_score(precision, got, want, ab[name].astype(np.float64).reshape(got.shape), floor), bank.kind + "." + name))
    loss = pop.loss[i].cpu().numpy().astype(np.float64)
    for k, key in enumerate(("critic_loss", "actor_loss")):
        items.append((abs(loss[k] - info[key]) / max(1.0, abs(info[key])) / LOSS_BAR[precision], key))
    return max(worst, max(x for x, _ in items))


def _step_score(got, before, want, names):
    """max over tensors of |(got - before) - (want - before)| / max|want - before| over UPD_BAR (<= 1 passes)."""
    worst = 0.0
    for n in names:
        b = before[n].astype(np.float64).reshape(-1)
        du, dw = got[n].astype(np.float64).reshape(-1) - b, want[n].astype(np.float64).reshape(-1) - b
        worst = max(worst, float(np.max(np.abs(du - dw)) / max(np.max(np.abs(dw)), 1e-30)) / UPD_BAR)
    return worst


def _named(bank, i):
    return {n: bank.view(n, i).cpu().numpy().copy() for n in bank.weight_names}


def _apply_scores(pop, i, before, grads, hp, step=1):
    """Scores of agent i's Adam step (both nets) and Polyak step (both targets) against oracle adam_apply + polyak run with the
    hyperparameters hp on the gradients `grads` (actor, critic dicts)."""
    scores = []
    for bank, tbank, g, lr, train, allw in ((pop.actor, pop.t_actor, grads[0], hp["actor_lr"], D.ACTOR_TRAINABLE, D.ACTOR_WEIGHTS),
                                            (pop.critic, pop.t_critic, grads[1], hp["critic_lr"], D.CRITIC_TRAINABLE, D.CRITIC_WEIGHTS)):
        p0, t0 = before[bank.kind], before["t_" + bank.kind]
        want = {k: v.copy() for k, v in p0.items()}
        m = {k: np.zeros_like(p0[k]) for k in train}
        v = {k: np.zeros_like(p0[k]) for k in train}
        D.adam_apply(want, g, m, v, step, lr, train)
        got = _named(bank, i)
        scores.append(_step_score(got, p0, want, train))
        want_t = D.polyak(t0, got, hp["tau"], allw)        # the targets follow the online weights the GPU produced
        scores.append(_step_score(_named(tbank, i), t0, want_t, allw))
    return max(scores)


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
def test_sweep_learn_step_vs_oracle(precision):
    """avd_ddpg_learn with apply_updates = 1 and a per-agent table (gamma 0.5 / 0.9 / 0.99, learning rates 10x apart, tau 1e-3 / 0.05
    / 0.5): every agent's gradients and losses against oracle.learn with its own gamma, its Adam and Polyak steps against
    oracle.adam_apply + polyak with its own learning rates and tau (on the gradients the step produced), at the bars of DESIGN.md
    section 4.  The same comparison with any other agent's value of one hyperparameter must fail its bar by 10x or more."""
    _need_gpu()
    from avddpg_b200.trainer import DDPGPopulation
    A, R = 3, 1000
    pop = DDPGPopulation(A, 1, _conf(), rows_per_agent=R, precision=precision, seeds=[11, 11, 12], overrides=HP3)
    assert pop.hp is not None and pop.hp.shape == (A, 4)
    nets = [_nets(50 + i) for i in range(A)]
    for four in nets:      # a target Q that dominates the TD target, so that gamma 0.9 against 0.99 moves the critic loss well past its bar
        four[3]["W3"] *= 20 if precision == 1 else 50         # (bf16 operands: less, their rounding of that larger Q counts too)
    for i, four in enumerate(nets):
        for bank, net in zip((pop.actor, pop.critic, pop.t_actor, pop.t_critic), four):
            bank.load_named(i, net)
    batches = [_batch(150 + i, R) for i in range(A)]
    cat = lambda j, w: torch.as_tensor(np.concatenate([b[j].reshape(R, w) for b in batches]), device="cuda").contiguous()
    before = [{"actor": _named(pop.actor, i), "critic": _named(pop.critic, i), "t_actor": _named(pop.t_actor, i),
               "t_critic": _named(pop.t_critic, i)} for i in range(A)]
    pop.learn(cat(0, 4), cat(1, 1).reshape(-1), cat(2, 1).reshape(-1), cat(3, 4), apply_updates=True)
    torch.cuda.synchronize()
    assert pop.actor.step.tolist() == [1] * A and pop.critic.step.tolist() == [1] * A
    margins = []
    for i in range(A):
        grads = ({n: pop.actor.view(n, i, pop.actor.grad).cpu().numpy() for n in pop.actor.trainable_names},
                 {n: pop.critic.view(n, i, pop.critic.grad).cpu().numpy() for n in pop.critic.trainable_names})
        items = []
        assert _learn_score(precision, pop, i, nets[i], batches[i], HP3[i]["gamma"], items) <= 1.0, (i, sorted(items)[-3:])
        assert _apply_scores(pop, i, before[i], grads, HP3[i]) <= 1.0, i
        for j in range(A):
            if j == i:
                continue
            margins.append(_learn_score(precision, pop, i, nets[i], batches[i], HP3[j]["gamma"]))
            for key in ("actor_lr", "critic_lr", "tau"):
                margins.append(_apply_scores(pop, i, before[i], grads, {**HP3[i], key: HP3[j][key]}))
    print(f"sweep learn precision={precision}: a misrouted value fails its bar by >= {min(margins):.0f}x")
    assert min(margins) >= 10.0, min(margins)


# ------------------------------------------------------------------------------------------ 3. fused FRL apply
@pytest.mark.parametrize("fused", [True, False])
def test_sweep_frl_apply_vs_oracle(fused):
    """A gradients round at world 1 over a population of two runs (interfrl: systems (follower, run), members the run's groups):
    fused, avd_fed_apply_gradients; unfused, reduce -> finalize -> broadcast -> apply_gradients_and_soft_update.  Every member's Adam
    and Polyak steps against the oracle with its run's learning rates and tau, on the system's averaged gradient."""
    _need_gpu()
    from avddpg_b200.server.federated import FederatedAggregator
    from avddpg_b200.trainer import DDPGPopulation
    Gr, S, M, R = 2, 2, 2, 64
    G, A = Gr * S, Gr * S * M
    conf = _conf(fed_method="interfrl")
    over = [HP3[0], HP3[2]]
    pop = DDPGPopulation(G, M, conf, rows_per_agent=R, precision=0, seeds=[5, 6], overrides=over)
    for a in range(A):
        four = _nets(70 + a)
        for bank, net in zip((pop.actor, pop.critic, pop.t_actor, pop.t_critic), four):
            bank.load_named(a, net)
    batches = [_batch(170 + a, R) for a in range(A)]
    cat = lambda j, w: torch.as_tensor(np.concatenate([b[j].reshape(R, w) for b in batches]), device="cuda").contiguous()
    pop.learn(cat(0, 4), cat(1, 1).reshape(-1), cat(2, 1).reshape(-1), cat(3, 4), apply_updates=False)
    ag0, cg0 = _np(pop.actor.grad).copy(), _np(pop.critic.grad).copy()
    before = [{"actor": _named(pop.actor, a), "critic": _named(pop.critic, a), "t_actor": _named(pop.t_actor, a),
               "t_critic": _named(pop.t_critic, a)} for a in range(A)]
    agg = FederatedAggregator(pop, conf, runs=S)
    if fused:
        assert agg.aggregate_gradients(apply=True, write_back=False) is None
    else:
        agg.aggregate_gradients(apply=False)
        pop.apply_gradients_and_soft_update()
    torch.cuda.synchronize()
    assert pop.actor.step.tolist() == [1] * A
    margins = []
    for a in range(A):
        m, g = divmod(a, G)
        run = g // Gr
        rows = [m * G + run * Gr + x for x in range(Gr)]
        ga, gc = ag0[rows].mean(0), cg0[rows].mean(0)
        grads = ({n: pop.actor.view(n, 0, torch.as_tensor(ga).unsqueeze(0)).numpy() for n in pop.actor.trainable_names},
                 {n: pop.critic.view(n, 0, torch.as_tensor(gc).unsqueeze(0)).numpy() for n in pop.critic.trainable_names})
        assert _apply_scores(pop, a, before[a], grads, over[run]) <= 1.0, (a, run)
        for key in ("actor_lr", "critic_lr", "tau"):
            margins.append(_apply_scores(pop, a, before[a], grads, {**over[run], key: over[1 - run][key]}))
    assert min(margins) >= 10.0, min(margins)
    with pytest.raises(NotImplementedError):
        pop.apply_gradients()
    with pytest.raises(NotImplementedError):
        pop.soft_update()


# ------------------------------------------------------------------------------------------ 4. closed loop
SWEEP3 = ([3, 5, 3], [dict(gamma=0.9, critic_lr=1e-3), dict(tau=0.002, std_dev=0.03), dict(actor_lr=1e-4, theta=0.2)])


@pytest.mark.parametrize("precision", [0, 2])
@pytest.mark.parametrize("fed", list(FED))
def test_sweep_closed_loop_with_learning(precision, fed):
    """50 steps of the full training step; every run against its stand-alone trainer built from run_config(s)."""
    _need_gpu()
    Gr, E, M = 2, 2, 2
    seeds, over = SWEEP3
    conf = _conf(pl_size=M, batch_size=16, buffer_size=64, can_terminate=False, episode_sim_time=1.0, **FED[fed])
    tr, alone = _sweep(conf, Gr, E, seeds, over, ring_capacity=64, precision=precision)
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
    print(f"sweep closed loop precision={precision} fed={fed}: states {worst_state:.1e} losses {worst_loss:.1e} weight updates {worst_upd:.1e}")
    assert worst_state < st_tol, worst_state
    assert worst_loss < loss_tol, worst_loss
    assert worst_upd < upd_tol, worst_upd
    # runs 0 and 2 share a seed and initial weights: their different hyperparameters must have taken them apart
    a0, a2 = tr.pop.run_agents(0).to(tr.pop.device), tr.pop.run_agents(2).to(tr.pop.device)
    assert not torch.equal(tr.pop.actor.flat[a0], tr.pop.actor.flat[a2])


# ------------------------------------------------------------------------------------------ 5. episode loop
def test_sweep_episode_loop(tmp_path):
    """run() per run with overrides: episode lengths, reward logs, Adam step counts and final weights against each run's stand-alone
    run(); every RewardLog carries its run's configuration, and two runs of one seed write files of the same names."""
    _need_gpu()
    seeds = [4, 21, 4]
    over = [dict(actor_lr=1e-4, gamma=0.9), dict(std_dev=0.03, theta=0.2), dict(critic_lr=1e-3, tau=0.002, std_dev=0.01)]
    conf = _conf(pl_size=2, batch_size=16, buffer_size=256, can_terminate=True, reset_ep_max=0.5, reset_max_ev=0.5, max_ep=1.0,
                 max_ev=1.0, episode_sim_time=3.0, fed_method="normal", reward_averaging_window=2)
    tr, alone = _sweep(conf, 1, 2, seeds, over, ring_capacity=256, precision=0)
    w0 = {b: _np(getattr(tr.pop, b).flat).astype(np.float64) for b in ("actor", "critic")}
    logs = tr.reward_logs()
    for k, log in enumerate(logs):
        assert log.conf.random_seed == seeds[k]
        for key, v in over[k].items():
            assert getattr(log.conf, key) == v, (k, key)
        for key in {"actor_lr", "critic_lr", "gamma", "tau", "std_dev", "theta"} - set(over[k]):
            assert getattr(log.conf, key) == getattr(conf, key), (k, key)
    episodes = 4
    tr.run(episodes, reward_logs=logs, learn=True)
    _, loss_tol, upd_tol = BARS[0]
    names = []
    for k, st in enumerate(alone):
        margins = _margin_recorder(st, conf)
        log = st.reward_logs()[0]
        lengths = [st.run(1, log, learn=True) for _ in range(episodes)]
        assert min(margins) > 1e-4, f"run {k}: a state came within {min(margins):.1e} of a terminal threshold"
        assert tr.run_episode_steps[k] == lengths, (k, tr.run_episode_steps[k], lengths)
        got, want = np.asarray(logs[k].all_ep_reward_lists, np.float64), np.asarray(log.all_ep_reward_lists, np.float64)
        assert got.shape == want.shape and np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-3)) < loss_tol, k
        agents = tr.pop.run_agents(k).to(tr.pop.device)
        assert int(st.pop.actor.step[0]) > 0, "learning must be active"
        assert torch.equal(tr.pop.actor.step[agents], st.pop.actor.step), k
        for b in ("actor", "critic"):
            g, w = _np(getattr(tr.pop, b).flat[agents]), _np(getattr(st.pop, b).flat)
            for a in range(g.shape[0]):
                assert _rel_update(g[a].astype(np.float64), w[a].astype(np.float64), w0[b][agents[a].item()]) < upd_tol, (k, b, a)
        out = tmp_path / f"run{k}"
        out.mkdir()
        names.append(sorted(p.split("/")[-1] for p in logs[k].generate_csvs(str(out))))
    assert names[0] == names[2] and names[0] != names[1], names


# ------------------------------------------------------------------------------------------ 6. graph capture
@pytest.mark.parametrize("learn", [False, True])
def test_sweep_graph_capture(learn):
    """A captured sweep trainer: 10 replays (20 steps) against 20 eager steps of a second trainer with the same seeds and overrides."""
    _need_gpu()
    from avddpg_b200.trainer import BatchedTrainer
    from test_gpu_runs import _capture_without_learning
    seeds = [5, 6, 5, 1 << 33]
    over = [dict(actor_lr=1e-3), dict(gamma=0.9, tau=0.05), dict(std_dev=0.05, theta=0.3, critic_lr=5e-3), {}]
    conf = _conf(pl_size=2, batch_size=16, buffer_size=64, can_terminate=True, max_ep=2.5, max_ev=2.5, episode_sim_time=2.0,
                 fed_method="interfrl", weighted_average_enabled=False)
    kw = dict(ring_capacity=64, precision=2, seeds=seeds, overrides=over)
    a, b = BatchedTrainer(conf, 2, 2, **kw), BatchedTrainer(conf, 2, 2, **kw)
    for tr in (a, b):
        for _ in range(20):
            tr.step(learn=learn)
    graph = a.capture(warmup=1) if learn else _capture_without_learning(a)
    b.step(learn=learn)
    for _ in range(10):
        graph.replay()
        b.step(learn=learn)
        b.step(learn=learn)
    torch.cuda.synchronize()
    assert torch.equal(a.env.episode, b.env.episode)
    written = min(a.rings.clock.read()["ring_count"], a.rings.capacity)
    if not learn:
        for name, x, y in (("obs", a.env.obs, b.env.obs), ("ring", a.rings.data[:written], b.rings.data[:written]), ("ou", a.env.ou_state, b.env.ou_state),
                           ("actions", a.env.action_out, b.env.action_out), ("ep_reward", a.env.ep_reward, b.env.ep_reward)):
            assert torch.equal(x, y), name
        return
    st_tol, loss_tol, _ = BARS[2]
    x, y = _np(a.env.obs).astype(np.float64), _np(b.env.obs).astype(np.float64)
    assert np.max(np.abs(x - y)) / np.max(np.abs(y)) < st_tol
    x, y = _np(a.rings.data[:written]).astype(np.float64), _np(b.rings.data[:written]).astype(np.float64)
    assert np.max(np.abs(x - y)) / np.max(np.abs(y)) < st_tol
    la, lb = _np(a.pop.loss).astype(np.float64), _np(b.pop.loss).astype(np.float64)
    assert np.max(np.abs(la - lb) / np.maximum(np.abs(lb), 1e-3)) < loss_tol
    assert torch.equal(a.pop.actor.step, b.pop.actor.step)


# ------------------------------------------------------------------------------------------ 7. refusals
def test_sweep_refusals():
    _need_gpu()
    import math
    from avddpg_b200.trainer import BatchedTrainer, DDPGPopulation
    ok = _conf(pl_size=2, batch_size=16, buffer_size=64)
    for kw in (dict(seeds=[1, 2], overrides=[{"batch_size": 32}, {}]), dict(seeds=[1, 2], overrides=[{}, {"pl_size": 3}]),
               dict(seeds=[1], overrides=[{"gamma": math.nan}]), dict(seeds=[1], overrides=[{"std_dev": math.inf}]),
               dict(seeds=[1, 2], overrides=[{}]), dict(overrides=[{}])):
        with pytest.raises(ValueError):
            BatchedTrainer(ok, 1, 1, ring_capacity=64, **kw)
    with pytest.raises(ValueError):
        BatchedTrainer(ok, 1, 1, ring_capacity=64, seeds=[1, 2], overrides=[{}, {"gamma": 0.5}], world=2)
    with pytest.raises(NotImplementedError):
        BatchedTrainer(_conf(pl_size=2, batch_size=16, buffer_size=64, fed_method="interfrl", aggregation_method="weights"), 1, 1,
                       ring_capacity=64, seeds=[1, 2], overrides=[{}, {"gamma": 0.5}])
    with pytest.raises(ValueError):
        DDPGPopulation(2, 1, ok, overrides=[{}, {}])
    pop = DDPGPopulation(2, 1, ok, seeds=[1, 2], overrides=[{}, {"tau": 0.1}])
    for call in (pop.apply_gradients, pop.soft_update):
        with pytest.raises(NotImplementedError):
            call()
    plain = BatchedTrainer(ok, 1, 1, ring_capacity=64, seeds=[1, 2])     # seeds only: no table anywhere
    assert plain.pop.hp is None and plain.runs.ou_sigma is None and plain.runs.table.ou_sigma is None
