"""GPU tests of the actor and critic forward passes (avd_actor_forward, avd_critic_forward, DDPGPopulation.act, evaluator.run) at
every precision, against the float64 evaluation of oracle/forward_bounds.py.

Every call checks three things:
  * the per-row bound of oracle/forward_bounds.row_bound holds on every row (a first-order worst case for the path that runs);
  * the normwise error max |got - exact| / max |exact| over the call's rows meets the bar of its precision:
      - precision 0 and 3: 1e-5, the bar of the fp32 parity tests;
      - precision 1 and 2: 2 E_model + 1e-5, where E_model is the normwise error of tools/precision_model.Net on the same
        inputs with the operands of the path that runs rounded (forward_bounds.model_sites).  The kernel rounds the same
        operands, so it should land on E_model up to fp32 accumulation order; 1e-5 (the fp32 bar) is the floor for that.
        On the CPU model at the weights used here E_model is 1e-4 to 4e-4 for fp16 and 1e-3 to 3.5e-3 for bf16; rounding
        r1 or W2' to bf16 at precision 2, or dropping the lo half of the split layer 1, gives 5 to 20 times E_model
        (tests/test_forward_bounds_cpu.py), so this bar rejects each of them.
        Measured on one B200 (1000 W power limit), worst over every call in this file: kernel error / E_model = 1.00 at
        precision 1 (fused and unfused) and at precision 2 unfused, 1.07 at precision 2 fused; largest normwise errors
        9.5e-3 (p1 fused), 1.1e-3 (p2 fused), 4.0e-3 (p1 / p2 unfused, bf16), 1.9e-6 (p0), 1.7e-6 (p3).  The kernel's
        error uses at most 1.5e-2 of the per-row bound on any row.
  * |action| <= action_high.
Around every call the output sits between two 64-float guards holding a NaN with a distinctive payload, the workspace is
exactly avd_forward_workspace_bytes with a guard behind it, and the weights and inputs are compared bit for bit afterwards.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ddpg_np as D
from oracle import forward_bounds as FB

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import precision_model as PM  # noqa: E402

pytestmark = pytest.mark.gpu

HIGH = 2.5
GUARD = 64
SENTINEL = 0x7FC0BEEF                         # a quiet NaN no kernel computes, as int32
WS_GUARD = 256
FP32_BAR = 1e-5
STD = (4, 256, 48, 128)                    # (ns, l1, la, l2) of the reference networks

# act() shapes of bench.py's configurations, by value: c2 = (G=1, E=4096, M=4), c4 = (G=1, E=8192, M=8)
ACT_SHAPES = [(1, 4096, 4), (1, 8192, 8), (3, 129, 3)]


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from avddpg_b200 import _lib, model, trainer
    from avddpg_b200.config import Config
    sm = _lib.require_device()[0]
    return dict(lib=_lib, model=model, trainer=trainer, Config=Config, sm=sm)


def make_nets(seed, dims=STD):
    """Actor and critic with non-trivial BatchNorm, biases and head weights (the generator of tests/test_gpu_ddpg.py)."""
    ns, l1, la, l2 = dims
    rng = np.random.default_rng(seed)
    ac, cr = D.init_actor(rng, ns, l1, l2), D.init_critic(rng, ns, l1, la, l2)
    D.randomize_bn(ac, rng, [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
    D.randomize_bn(cr, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")])
    for p in (ac, cr):
        for k in p:
            if k.startswith("b") and not k.startswith("be"):
                p[k] = rng.normal(0, 0.05, p[k].shape).astype(np.float32)
    ac["W3"] *= 50
    cr["W3"] *= 300
    return ac, cr


def make_bank(mods, kind, dims, nets):
    bank = mods["model"].NetBank(kind, mods["model"].make_dims(*dims), len(nets), "cuda")
    for i, p in enumerate(nets):
        bank.load_named(i, p)
    return bank


def guarded(n):
    buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda")
    return buf, buf[GUARD:GUARD + n].view(torch.float32)


def check_guards(buf, n):
    b = buf.cpu()
    assert (b[:GUARD] == SENTINEL).all() and (b[GUARD + n:] == SENTINEL).all(), "output guard overwritten"
    left = int((b[GUARD:GUARD + n] == SENTINEL).sum())
    assert left == 0, f"{left} of {n} outputs never written"


def call(mods, kind, dims, bank, A, R, s, s_rs, s_cs, a=None, precision=0):
    """One avd_actor_forward / avd_critic_forward with guarded output and an exact workspace; -> outputs [A*R] (float64)."""
    lib, L = mods["lib"], mods["lib"].load()
    d = mods["model"].make_dims(*dims)
    n = A * R
    need = L.avd_forward_workspace_bytes(C.byref(d), A, R, int(kind == "critic"), precision)
    assert need > 0
    ws = torch.full((need + WS_GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
    buf, out = guarded(n)
    before = [bank.flat.clone(), s.clone()] + ([a.clone()] if a is not None else [])
    if kind == "actor":
        lib.check(L.avd_actor_forward(C.byref(d), A, R, lib.ptr(bank.flat), lib.ptr(s), s_rs, s_cs, HIGH, lib.ptr(out), lib.ptr(ws),
                                      need, precision, lib.current_stream()))
    else:
        assert s_rs == dims[0] and s_cs == 1, "avd_critic_forward reads row-major states with pitch ns"
        lib.check(L.avd_critic_forward(C.byref(d), A, R, lib.ptr(bank.flat), lib.ptr(s), lib.ptr(a), lib.ptr(out), lib.ptr(ws), need,
                                       precision, lib.current_stream()))
    torch.cuda.synchronize()
    check_guards(buf, n)
    assert (ws[need:].cpu() == 0xA5).all(), "workspace guard overwritten"
    for t0, t1 in zip(before, [bank.flat, s] + ([a] if a is not None else [])):
        assert torch.equal(t0.view(torch.int32), t1.view(torch.int32)), "an input changed"
    return out.cpu().numpy().astype(np.float64)


def check_rows(kind, dims, precision, nets_of_agent, states, actions, got, tag=""):
    """Per-row bound, normwise bar and action range.  nets_of_agent: parameter dict per agent; states [A][R][ns]."""
    critic = kind == "critic"
    A = len(nets_of_agent)
    R = len(got) // A
    ref, bnd, model = np.empty(A * R), np.empty(A * R), np.empty(A * R)
    sites = FB.model_sites(dims, precision)
    for i, p in enumerate(nets_of_agent):
        s = np.asarray(states[i], np.float64)
        a = None if actions is None else np.asarray(actions[i], np.float64)
        rows = slice(i * R, (i + 1) * R)
        bnd[rows], ref[rows] = FB.row_bound(p, critic, s, a, dims=dims, precision=precision, high=HIGH)
        if precision in (1, 2):
            model[rows] = FB.output(PM.Net(p, critic, sites).forward(s, a)[0], critic, HIGH)
    err = np.abs(got - ref)
    bad = np.flatnonzero(~(err <= bnd))
    assert bad.size == 0, f"{tag}: {bad.size} rows outside the bound, first {bad[:5]}: err {err[bad[:5]]} bound {bnd[bad[:5]]}"
    e = FB.normwise(got, ref)
    if precision in (1, 2):
        em = FB.normwise(model, ref)
        assert e <= 2 * em + FP32_BAR, f"{tag}: normwise {e:.3e} above 2 x model {em:.3e} + {FP32_BAR}"
    else:
        assert e <= FP32_BAR, f"{tag}: normwise {e:.3e}"
    if not critic:
        assert np.all(np.abs(got) <= HIGH)


def rand_states(seed, n, ns, scale=2.0):
    rng = np.random.default_rng(seed)
    return rng.normal(0, scale, (n, ns)).astype(np.float32), rng.uniform(-HIGH, HIGH, n).astype(np.float32)


def run_case(mods, A, R, precision, dims=STD, seed=0, layout="rows"):
    """Actor and critic of A agents (distinct weights) on R rows each; actor states in the given layout."""
    ns = dims[0]
    nets = [make_nets(1000 * seed + i, dims) for i in range(A)]
    n = A * R
    s_np, a_np = rand_states(seed + 7, n, ns)
    s_rows = torch.as_tensor(s_np, device="cuda")
    a = torch.as_tensor(a_np, device="cuda")
    if layout == "rows":
        s, s_rs, s_cs = s_rows, ns, 1
    elif layout == "pitch5":            # odd pitch with a NaN in the unused word
        s = torch.full((n, 5), float("nan"), device="cuda")
        s[:, :ns] = s_rows
        s, s_rs, s_cs = s.reshape(-1), 5, 1
    elif layout == "native":            # [ns][N]: row stride 1, column stride N (the environment's [4][M][P] state)
        s, s_rs, s_cs = s_rows.t().contiguous(), 1, n
    else:
        raise ValueError(layout)
    st = s_np.reshape(A, R, ns)
    got = call(mods, "actor", dims, make_bank(mods, "actor", dims, [x[0] for x in nets]), A, R, s, s_rs, s_cs, precision=precision)
    check_rows("actor", dims, precision, [x[0] for x in nets], st, None, got, f"actor A={A} R={R} p{precision} {layout}")
    if layout == "rows":
        got = call(mods, "critic", dims, make_bank(mods, "critic", dims, [x[1] for x in nets]), A, R, s_rows, ns, 1, a, precision)
        check_rows("critic", dims, precision, [x[1] for x in nets], st, a_np.reshape(A, R), got, f"critic A={A} R={R} p{precision}")


SHAPES = [(2, 1), (2, 127), (2, 128), (2, 129), (3, 70), (2, 4133), (1, 100_003), (300, 5)]


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
@pytest.mark.parametrize("A,R", SHAPES)
def test_forward_shapes(mods, A, R, precision):
    run_case(mods, A, R, precision, seed=A + R)


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
@pytest.mark.parametrize("extra", [0, 1])
def test_forward_agents_around_sm_count(mods, extra, precision):
    """One CTA per agent once A reaches the SM count (ctas_per_agent), and more agents than SMs."""
    run_case(mods, mods["sm"] + extra, 64, precision, seed=5 + extra)


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
@pytest.mark.parametrize("layout", ["pitch5", "native"])
def test_actor_state_layouts(mods, layout, precision):
    """Row pitch 5 and the column-major native layout over several tiles and CTAs per agent (row-major pitch 4 is every
    other test)."""
    run_case(mods, 3, 1000, precision, seed=11, layout=layout)


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
def test_model_a_three_states_ignores_the_unused_word(mods, precision):
    """Model A: ns = 3.  Actor rows of 4 words whose 4th is NaN (a kernel that multiplies it by a zero weight returns NaN), and
    rows of pitch ns = 3 for both networks."""
    dims = (3, 256, 48, 128)
    A, R = 2, 300
    nets = [make_nets(40 + i, dims) for i in range(A)]
    s_np, a_np = rand_states(41, A * R, 3)
    s4 = torch.full((A * R, 4), float("nan"), device="cuda")
    s4[:, :3] = torch.as_tensor(s_np, device="cuda")
    s3 = torch.as_tensor(s_np, device="cuda")
    actor = make_bank(mods, "actor", dims, [x[0] for x in nets])
    for s, rs in ((s4, 4), (s3, 3)):
        got = call(mods, "actor", dims, actor, A, R, s, rs, 1, precision=precision)
        check_rows("actor", dims, precision, [x[0] for x in nets], s_np.reshape(A, R, 3), None, got, f"model A actor pitch {rs}")
    got = call(mods, "critic", dims, make_bank(mods, "critic", dims, [x[1] for x in nets]), A, R, s3, 3, 1,
               torch.as_tensor(a_np, device="cuda"), precision)
    check_rows("critic", dims, precision, [x[1] for x in nets], s_np.reshape(A, R, 3), a_np.reshape(A, R), got, "model A critic")


@pytest.mark.parametrize("precision", [1, 2])
@pytest.mark.parametrize("dims", [(4, 256, 48, 128), (4, 256, 56, 128), (4, 256, 64, 128), (5, 256, 48, 128), (4, 256, 48, 96),
                                  (4, 264, 48, 128)], ids=lambda d: "ns{}-l1{}-la{}-l2{}".format(*d))
def test_fused_unfused_boundary(mods, dims, precision):
    """Each side of fused3::supported (la <= 48, ns <= 4, l2 == 128, l1 == 256): outside it precision 1 and 2 both run the
    unfused GEMMs on bf16 operands, and the bar follows the path that runs."""
    run_case(mods, 2, 300, precision, dims=dims, seed=sum(dims))


def test_fp16_range(mods):
    """States x 3e4 at precision 2: layer-1 activations beyond the fp16 range saturate, outputs stay finite and in range."""
    A, R = 2, 300
    nets = [make_nets(90 + i) for i in range(A)]
    s_np, a_np = rand_states(91, A * R, 4)
    s = torch.as_tensor(s_np * 3e4, device="cuda")
    got = call(mods, "actor", STD, make_bank(mods, "actor", STD, [x[0] for x in nets]), A, R, s, 4, 1, precision=2)
    assert np.isfinite(got).all() and np.all(np.abs(got) <= HIGH)
    got = call(mods, "critic", STD, make_bank(mods, "critic", STD, [x[1] for x in nets]), A, R, s, 4, 1,
               torch.as_tensor(a_np, device="cuda"), 2)
    assert np.isfinite(got).all()


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
@pytest.mark.parametrize("G,E,M", ACT_SHAPES)
def test_population_act(mods, G, E, M, precision):
    """DDPGPopulation.act on the environment's native state [4][M][P], P = G E: row n = m P + p belongs to agent n // E."""
    conf = mods["Config"](pl_size=M)
    pop = mods["trainer"].DDPGPopulation(G, M, conf, precision=precision)
    A, P = G * M, G * E
    nets = [make_nets(300 + i)[0] for i in range(A)]
    for i, p in enumerate(nets):
        pop.actor.load_named(i, p)
    rng = np.random.default_rng(E + M)
    st = rng.normal(0, 2, (4, M, P)).astype(np.float32)
    native = torch.as_tensor(st, device="cuda")
    buf, out = guarded(M * P)
    w0 = pop.actor.flat.clone()
    pop.act(native, out.view(M, P), envs_per_group=E)
    torch.cuda.synchronize()
    check_guards(buf, M * P)
    assert torch.equal(w0, pop.actor.flat) and torch.equal(native, torch.as_tensor(st, device="cuda"))
    rows = st.reshape(4, M * P).T.reshape(A, E, 4)
    check_rows("actor", STD, precision, nets, rows, None, out.cpu().numpy().astype(np.float64), f"act G={G} E={E} M={M}")


@pytest.mark.parametrize("precision", [0, 1, 2, 3])
@pytest.mark.parametrize("kind", ["actor", "critic"])
def test_rows_are_independent(mods, kind, precision):
    """Each output row depends only on its own input row and its agent's weights, bit for bit: permuting an agent's rows
    permutes its outputs, appending 37 rows (the tile boundaries shift) leaves the first R outputs unchanged, and the same
    weights at agent 0 and agent 3 give the same outputs for the same rows.  (The folded layer-2 bias b2' of the tensor-core
    paths was once summed with atomics in CTA completion order, which broke the last of these by a few ulp.)"""
    A, R = 5, 300
    nets = [make_nets(500 + i) for i in range(A)]
    j = 0 if kind == "actor" else 1
    nets[3] = nets[0]
    bank = make_bank(mods, kind, STD, [x[j] for x in nets])
    s_np, a_np = rand_states(501, A * (R + 37), 4)
    s_np, a_np = s_np.reshape(A, R + 37, 4), a_np.reshape(A, R + 37)
    s_np[3], a_np[3] = s_np[0], a_np[0]

    def fwd(s, a, Rk):
        st = torch.as_tensor(np.ascontiguousarray(s).reshape(-1, 4), device="cuda")
        at = torch.as_tensor(np.ascontiguousarray(a).reshape(-1), device="cuda")
        out = call(mods, kind, STD, bank, A, Rk, st, 4, 1, at if kind == "critic" else None, precision)
        return out.reshape(A, Rk)

    base = fwd(s_np[:, :R], a_np[:, :R], R)
    assert np.array_equal(base[3], base[0]), "same weights and rows at agent 0 and agent 3"
    longer = fwd(s_np, a_np, R + 37)
    assert np.array_equal(longer[:, :R], base), "appending rows changed earlier outputs"
    perm = np.random.default_rng(7).permutation(R)
    permuted = fwd(s_np[:, perm], a_np[:, perm], R)
    assert np.array_equal(permuted, base[:, perm]), "permuting rows changed their outputs"


def test_evaluator_precision3_meets_the_fp32_bars(mods, golden):
    """evaluator.run at precision 3 on the reference's seed-6 inputs meets the precision-0 bars of
    test_gpu_ddpg.py::test_evaluator_rollout_vs_reference_golden."""
    from avddpg_b200 import evaluator
    g, conf, pop, T = _evaluator_setup(mods, golden)
    pl_rew, tr = evaluator.run(conf, pop, num_platoons=2, leader_inputs=np.repeat(g["inputs"][:, None], 2, axis=1),
                               manual_timestep_override=T, precision=3, return_traces=True)
    st = tr["states"].cpu().numpy()
    assert FB.normwise(st[:, 0], g["states"]) < 2e-5 and FB.normwise(tr["inputs"][:, 0].cpu().numpy(), g["actions"]) < 2e-5
    assert FB.normwise(tr["jerks"][:, 0].cpu().numpy(), g["jerks"]) < 5e-4
    np.testing.assert_allclose(tr["rewards"][0].cpu().numpy(), g["ep_reward"], rtol=2e-5)
    assert abs(pl_rew - float(g["pl_rew"])) <= 1e-3


def _model_action_error(g, precision):
    """Normwise error of tools/precision_model.py's actors at `precision` on the golden rollout's states (every vehicle)."""
    err, ref = [], []
    for m in range(3):
        p = {k[len(f"actor{m}_"):]: v for k, v in g.items() if k.startswith(f"actor{m}_")}
        s = np.asarray(g["states"][:, m, :], np.float64)
        r = FB.output(FB.exact(p, False, s)[0], False, HIGH)
        err.append(FB.output(PM.Net(p, False, FB.model_sites(STD, precision)).forward(s)[0], False, HIGH) - r)
        ref.append(r)
    return np.max(np.abs(np.concatenate(err))) / np.max(np.abs(np.concatenate(ref)))


@pytest.mark.parametrize("precision", [1, 2])
def test_evaluator_tensor_core_trajectory(mods, golden, precision):
    """The 100-step noise-free rollout at precision 2 stays within the closed-loop bar on states of tests/test_gpu_loop.py
    (5e-4 normwise).  Precision 1 is held to that bar times the ratio of the per-step action errors of the two precisions, which
    the CPU model gives on these actors and states (5.8: bf16 operands have 8 times the unit roundoff of fp16): the closed loop
    is linear in small action errors.  Measured on one B200 (1000 W): 8.9e-5 at precision 2, 1.1e-3 at precision 1 (bar 2.9e-3)."""
    from avddpg_b200 import evaluator
    g, conf, pop, T = _evaluator_setup(mods, golden)
    _, tr = evaluator.run(conf, pop, num_platoons=2, leader_inputs=np.repeat(g["inputs"][:, None], 2, axis=1),
                          manual_timestep_override=T, precision=precision, return_traces=True)
    st = tr["states"].cpu().numpy()
    assert np.isfinite(st).all()
    bar = 5e-4 * _model_action_error(g, precision) / _model_action_error(g, 2)
    assert FB.normwise(st[:, 0], g["states"]) < bar


def _evaluator_setup(mods, golden):
    g = golden("evaluator")
    conf = mods["Config"](pl_size=3)
    pop = mods["trainer"].DDPGPopulation(1, 3, conf)
    for m in range(3):
        pop.actor.load_named(m, {k[len(f"actor{m}_"):]: v for k, v in g.items() if k.startswith(f"actor{m}_")})
    return g, conf, pop, int(g["T"])

