"""precision = 3: the unfused tensor-core learn step on three-way split bf16 operands (avd_gemm_bf16x3), held to the bars of the
fp32 SIMT parity mode (precision = 0), not to looser ones.

  split GEMM alone      elementwise |C - C64| <= 2 K 2^-24 (|A| |B|), the fp32 dot-product bound
  forward               1e-5 normwise against oracle/ddpg_np.py
  gradients, losses     2e-4 normwise per gradient tensor, losses 1e-4 (Model A: 2e-4 condition-normalised)
  Adam + Polyak x3      rtol 2e-4, atol 2e-6
  closed loop (50 steps) states 2e-5, losses 1e-4, weight updates 5e-3 rel-L2 per tensor
"""
import numpy as np
import pytest
import torch

from oracle import ddpg_np as D
from oracle.loop_np import TrainLoopOracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from avddpg_b200 import _lib, trainer
    from avddpg_b200.config import Config
    _lib.require_device()
    return dict(lib=_lib, trainer=trainer, Config=Config)


def _nrm(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return np.max(np.abs(got - ref)) / max(np.max(np.abs(ref)), 1e-12)


def _nets(seed, la=48):
    rng = np.random.default_rng(seed)
    nets = [D.init_actor(rng), D.init_critic(rng, la=la), D.init_actor(rng), D.init_critic(rng, la=la)]
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


def _population(mods, A, R, seeds, la=48):
    conf = mods["Config"](critic_act_layer_size=la)
    pop = mods["trainer"].DDPGPopulation(A, 1, conf, rows_per_agent=R, precision=3)
    nets = [_nets(sd, la) for sd in seeds]
    for a, four in enumerate(nets):
        for bank, net in zip((pop.actor, pop.critic, pop.t_actor, pop.t_critic), four):
            bank.load_named(a, net)
    batches = [_batch(100 + sd, R) for sd in seeds]
    cat = lambda i, w: torch.as_tensor(np.concatenate([b[i].reshape(R, w) for b in batches]), device="cuda").contiguous()
    return conf, pop, nets, batches, (cat(0, 4), cat(1, 1).reshape(-1), cat(2, 1).reshape(-1), cat(3, 4))


# ------------------------------------------------------------------------------------------ the split GEMM alone
def _planes(x):
    """[..] fp32 -> [3, ..] bf16 planes hi, mid, lo (hi + mid + lo == x for every finite fp32 x of normal range)."""
    hi = x.bfloat16()
    r = x - hi.float()
    mid = r.bfloat16()
    lo = (r - mid.float()).bfloat16()
    return torch.stack([hi, mid, lo]).contiguous()


@pytest.mark.parametrize("layout,batch,M,N,K,splitk", [
    (0, 1, 128, 128, 64, 1), (0, 2, 200, 128, 272, 1), (0, 3, 70, 48, 304, 1), (0, 1, 1000, 304, 128, 1), (0, 1, 256, 128, 1024, 4),
    (1, 1, 304, 128, 1000, 4), (1, 2, 272, 48, 700, 3), (1, 3, 136, 128, 64, 1), (1, 2, 304, 128, 4096, 8), (1, 1, 256, 64, 333, 1)])
def test_split_gemm_meets_fp32_dot_product_bound(mods, layout, batch, M, N, K, splitk):
    lib = mods["lib"]
    g = torch.Generator(device="cuda").manual_seed(1000 * layout + M + 7 * N + K)
    if layout == 0:
        A = torch.randn(batch, M, K, device="cuda", generator=g)
        B = torch.randn(batch, N, K, device="cuda", generator=g)
        ref = torch.einsum("bmk,bnk->bmn", A.double(), B.double())
        bound = torch.einsum("bmk,bnk->bmn", A.double().abs(), B.double().abs())
        lda, ldb, a_batch, b_batch = K, K, M * K, N * K
    else:
        A = torch.randn(batch, K, M, device="cuda", generator=g)
        B = torch.randn(batch, K, N, device="cuda", generator=g)
        ref = torch.einsum("bkm,bkn->bmn", A.double(), B.double())
        bound = torch.einsum("bkm,bkn->bmn", A.double().abs(), B.double().abs())
        lda, ldb, a_batch, b_batch = M, N, K * M, K * N
    Ap, Bp = _planes(A), _planes(B)
    C = torch.zeros(batch, M, N, device="cuda")
    lib.check(lib.load().avd_gemm_bf16x3(layout, batch, M, N, K, lib.ptr(Ap), lda, a_batch, lib.ptr(Bp), ldb, b_batch, lib.ptr(C), N, M * N,
                                         splitk, lib.current_stream()))
    torch.cuda.synchronize()
    excess = ((C.double() - ref).abs() - 2 * K * 2.0 ** -24 * bound).max().item()
    assert excess <= 0, excess
    # Normwise, against the product of two-term (hi + mid) operands: losing any one of the 2^-16-order products hi.lo, mid.mid,
    # lo.hi costs about a third of that error or more, so the bar below catches it where the worst-case bound above does not.
    two = lambda P: P[0].double() + P[1].double()
    x2 = torch.einsum("bmk,bnk->bmn" if layout == 0 else "bkm,bkn->bmn", two(Ap), two(Bp))
    err, err_x2 = ((C.double() - ref).norm() / ref.norm()).item(), ((x2 - ref).norm() / ref.norm()).item()
    assert err < err_x2 / 4, (err, err_x2)


# ------------------------------------------------------------------------------------------ forward passes
@pytest.mark.parametrize("A,R", [(3, 70), (2, 300)])
def test_forward_vs_oracle(mods, A, R):
    conf, pop, nets, batches, (s, a, r, s2) = _population(mods, A, R, list(range(71, 71 + A)))
    lib, d = mods["lib"], pop.dims
    n = A * R
    out = torch.empty(n, device="cuda"); q = torch.empty(n, device="cuda")
    ws_a = lib.load().avd_forward_workspace_bytes(d, A, R, 0, 3)
    ws_c = lib.load().avd_forward_workspace_bytes(d, A, R, 1, 3)
    assert ws_a > lib.load().avd_forward_workspace_bytes(d, A, R, 0, 1)
    ws = torch.empty(max(ws_a, ws_c), dtype=torch.uint8, device="cuda")
    lib.check(lib.load().avd_actor_forward(d, A, R, lib.ptr(pop.actor.flat), lib.ptr(s), 4, 1, 2.5, lib.ptr(out), lib.ptr(ws), ws_a, 3,
                                           lib.current_stream()))
    lib.check(lib.load().avd_critic_forward(d, A, R, lib.ptr(pop.critic.flat), lib.ptr(s), lib.ptr(a), lib.ptr(q), lib.ptr(ws), ws_c, 3,
                                            lib.current_stream()))
    torch.cuda.synchronize()
    for i in range(A):
        ref_a, _ = D.actor_forward(nets[i][0], batches[i][0])
        ref_q, _ = D.critic_forward(nets[i][1], batches[i][0], batches[i][1])
        assert _nrm(out[i * R:(i + 1) * R].cpu().numpy(), ref_a.ravel()) < 1e-5
        assert _nrm(q[i * R:(i + 1) * R].cpu().numpy(), ref_q.ravel()) < 1e-5


# ------------------------------------------------------------------------------------------ gradients and losses
def _check_learn(mods, pop, nets, batches, conf, A):
    bad = []
    for i in range(A):
        ocg, oag, info = D.learn(nets[i][0], nets[i][1], nets[i][2], nets[i][3], batches[i], gamma=conf.gamma, high=conf.action_high)
        for bank, ref in ((pop.critic, ocg), (pop.actor, oag)):
            for name in bank.trainable_names:
                got = bank.view(name, i, bank.grad).cpu().numpy()
                e = _nrm(got, ref[name].reshape(got.shape))
                if not e < 2e-4:
                    bad.append((i, bank.kind, name, float(e)))
        loss = pop.loss[i].cpu().numpy()
        for k, key in enumerate(("critic_loss", "actor_loss")):
            if not abs(loss[k] - info[key]) < 1e-4 * max(1, abs(info[key])):
                bad.append((i, key, float(loss[k]), float(info[key])))
    assert not bad, bad


@pytest.mark.parametrize("A,R", [(1, 64), (3, 64), (2, 200), (2, 1000), (200, 64), (3, 100_003), (1, 250_000)])
def test_learn_gradients_vs_oracle(mods, A, R):
    """(200, 64): more agents than SMs; (3, 100003): ragged last row tile and many split-K CTAs of the weight-gradient GEMM."""
    conf, pop, nets, batches, (s, a, r, s2) = _population(mods, A, R, list(range(10, 10 + A)))
    pop.learn(s, a, r, s2, apply_updates=False)
    torch.cuda.synchronize()
    _check_learn(mods, pop, nets, batches, conf, A)


@pytest.mark.parametrize("la", [16, 32, 64])
def test_learn_other_action_layer_sizes(mods, la):
    """la = 16: K = l1 + la = 272 ends in a partial K block; la = 64 is a width the fused kernels do not take."""
    A, R = 2, 700
    conf, pop, nets, batches, (s, a, r, s2) = _population(mods, A, R, [90 + la, 91 + la], la=la)
    assert pop.dims.la == la
    pop.learn(s, a, r, s2, apply_updates=False)
    torch.cuda.synchronize()
    _check_learn(mods, pop, nets, batches, conf, A)


def test_learn_three_state_model_a(mods):
    """Model A: dims.ns = 3 read out of 4-word rows (s_stride 4) whose unused word holds garbage."""
    conf = mods["Config"](model="ModelA")
    R = 1000
    pop = mods["trainer"].DDPGPopulation(1, 1, conf, num_states=3, rows_per_agent=R, precision=3)
    rng = np.random.default_rng(3)
    nets = [D.init_actor(rng, ns=3), D.init_critic(rng, ns=3), D.init_actor(rng, ns=3), D.init_critic(rng, ns=3)]
    nets[0]["W3"] *= 50; nets[1]["W3"] *= 300; nets[2]["W3"] *= 50; nets[3]["W3"] *= 300
    for bank, net in zip((pop.actor, pop.critic, pop.t_actor, pop.t_critic), nets):
        bank.load_named(0, net)
    s, a, r, s2 = _batch(5, R)
    s3, s23 = s[:, :3].copy(), s2[:, :3].copy()
    s[:, 3], s2[:, 3] = 1e3, -1e3
    dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), device="cuda")
    pop.learn(dev(s), dev(a.reshape(-1)), dev(r.reshape(-1)), dev(s2), apply_updates=False)
    torch.cuda.synchronize()
    ocg, oag, info = D.learn(nets[0], nets[1], nets[2], nets[3], (s3, a, r, s23), gamma=conf.gamma, high=conf.action_high, with_abs=True)
    for bank, ref, ab in ((pop.critic, ocg, info["critic_abs"]), (pop.actor, oag, info["actor_abs"])):
        for name in bank.trainable_names:
            got = bank.view(name, 0, bank.grad).cpu().numpy().astype(np.float64)
            want = ref[name].reshape(got.shape).astype(np.float64)
            err = np.linalg.norm(got - want) / max(np.linalg.norm(ab[name].astype(np.float64)), 1e-300)
            assert err < 2e-4, (bank.kind, name, err)


def test_learn_apply_updates_sequence(mods):
    """Three consecutive local updates (Adam x2 + Polyak) stay on the oracle's trajectory."""
    A, R = 2, 64
    conf, pop, nets, batches, (s, a, r, s2) = _population(mods, A, R, [21, 22])
    state = []
    for ac, cr, ta, tc in nets:
        z = lambda p, names: {k: np.zeros_like(p[k]) for k in names}
        state.append(dict(am=z(ac, D.ACTOR_TRAINABLE), av=z(ac, D.ACTOR_TRAINABLE), cm=z(cr, D.CRITIC_TRAINABLE), cv=z(cr, D.CRITIC_TRAINABLE)))
    for step in range(1, 4):
        pop.learn(s, a, r, s2, apply_updates=True)
        for i, (ac, cr, ta, tc) in enumerate(nets):
            ocg, oag, _ = D.learn(ac, cr, ta, tc, batches[i], gamma=conf.gamma, high=conf.action_high)
            D.adam_apply(cr, ocg, state[i]["cm"], state[i]["cv"], step, conf.critic_lr, D.CRITIC_TRAINABLE)
            D.adam_apply(ac, oag, state[i]["am"], state[i]["av"], step, conf.actor_lr, D.ACTOR_TRAINABLE)
            nets[i][3] = tc = D.polyak(tc, cr, conf.tau, D.CRITIC_WEIGHTS)
            nets[i][2] = ta = D.polyak(ta, ac, conf.tau, D.ACTOR_WEIGHTS)
    torch.cuda.synchronize()
    assert pop.actor.step.tolist() == [3, 3] and pop.critic.step.tolist() == [3, 3]
    for i, (ac, cr, ta, tc) in enumerate(nets):
        for bank, ref in ((pop.actor, ac), (pop.critic, cr), (pop.t_actor, ta), (pop.t_critic, tc)):
            for name in bank.weight_names:
                got = bank.view(name, i).cpu().numpy()
                np.testing.assert_allclose(got, ref[name].reshape(got.shape), rtol=2e-4, atol=2e-6, err_msg=f"{bank.kind}.{name}")


# ------------------------------------------------------------------------------------------ the whole training step
@pytest.mark.parametrize("fed", [None, "interfrl", "intrafrl"])
def test_closed_loop_parity(mods, fed):
    """50 steps of BatchedTrainer(precision=3) beside oracle.loop_np.TrainLoopOracle (same weights, same counter-based draws)."""
    G, E, M, K = 2, 4, 2, 50
    conf = mods["Config"](pl_size=M, batch_size=16, buffer_size=64, can_terminate=False, fed_method=fed or "normal", weighted_average_enabled=False)
    tr = mods["trainer"].BatchedTrainer(conf, num_groups=G, envs_per_group=E, ring_capacity=64, precision=3)
    rng = np.random.default_rng(7)
    nets = []
    for _ in range(M * G):
        ac, cr = D.init_actor(rng), D.init_critic(rng)
        D.randomize_bn(ac, rng, [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
        D.randomize_bn(cr, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")])
        ac["W3"] *= 50
        cr["W3"] *= 100
        nets.append([ac, cr, {k: v.copy() for k, v in ac.items()}, {k: v.copy() for k, v in cr.items()}])
    for a, four in enumerate(nets):
        for bank, net in zip((tr.pop.actor, tr.pop.critic, tr.pop.t_actor, tr.pop.t_critic), four):
            bank.load_named(a, net)
    ora = TrainLoopOracle(conf, G, E, M, nets, seed=tr.env.seed, ring_capacity=64, fed=fed)
    worst_state = worst_loss = 0.0
    n_learn = 0
    for k in range(K):
        tr.step()
        obs, rew, _ = ora.step()
        got = tr.env.obs.cpu().numpy().astype(np.float64)
        worst_state = max(worst_state, float(np.max(np.abs(got - obs)) / np.max(np.abs(obs))))
        assert np.max(np.abs(tr.env.reward.cpu().numpy() - rew)) < 5e-5 + 10 * 2e-5, k
        if ora.count > ora.batch:
            n_learn += 1
            loss = tr.pop.loss.cpu().numpy().astype(np.float64)
            want = np.asarray(ora.losses[-1], dtype=np.float64)
            worst_loss = max(worst_loss, float(np.max(np.abs(loss - want) / np.maximum(np.abs(want), 1e-3))))
    assert n_learn == K - 16 and tr.pop.actor.step.tolist() == [n_learn] * (M * G)
    assert worst_state < 2e-5, worst_state
    assert worst_loss < 1e-4, worst_loss
    worst_upd, where = 0.0, None
    for a in range(M * G):
        for bank, ref, init, names in ((tr.pop.actor, ora.nets[a][0], nets[a][0], D.ACTOR_TRAINABLE), (tr.pop.critic, ora.nets[a][1], nets[a][1], D.CRITIC_TRAINABLE),
                                       (tr.pop.t_actor, ora.nets[a][2], nets[a][2], D.ACTOR_WEIGHTS), (tr.pop.t_critic, ora.nets[a][3], nets[a][3], D.CRITIC_WEIGHTS)):
            for name in names:
                got = bank.view(name, a).cpu().numpy().astype(np.float64).ravel()
                want, w0 = ref[name].astype(np.float64).ravel(), init[name].astype(np.float64).ravel()
                upd = np.linalg.norm(want - w0)
                if upd < 1e-5 * max(np.linalg.norm(w0), 1e-30):      # never trained (BatchNorm moving statistics)
                    assert np.linalg.norm(got - want) <= 5e-6 * np.linalg.norm(w0), (a, bank.kind, name)
                    continue
                e = float(np.linalg.norm(got - want) / upd)
                if e > worst_upd:
                    worst_upd, where = e, (a, bank.kind, name)
    assert worst_upd < 5e-3, (worst_upd, where)
    print(f"closed loop precision=3 fed={fed}: states {worst_state:.1e} losses {worst_loss:.1e} weight updates {worst_upd:.1e} at {where}")


def test_graph_capture_and_replay(mods):
    conf = mods["Config"](pl_size=2, batch_size=8, buffer_size=64)
    tr = mods["trainer"].BatchedTrainer(conf, num_groups=2, envs_per_group=40, ring_capacity=64, precision=3)
    for _ in range(14):
        tr.step()
    torch.cuda.synchronize()
    w0 = tr.pop.critic.flat.clone()
    tr.capture(warmup=1)
    tr.replay()
    torch.cuda.synchronize()
    assert not torch.equal(w0, tr.pop.critic.flat)
    for t in (tr.pop.actor.flat, tr.pop.critic.flat, tr.pop.t_actor.flat, tr.pop.t_critic.flat, tr.pop.loss):
        assert torch.isfinite(t).all()
