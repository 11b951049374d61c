"""Time and accuracy of the learn call at the C2 learn shape (4 agents x 262,144 rows) for precision 0 (fp32 SIMT parity kernels),
2 (fp16 tensor-core operands, the bench default) and 3 (three-way split bf16 operands on tcgen05), in one process.

    python tools/bench_precision.py [--out profiles/r03_precision3.json] [--rows 262144] [--calls 30] [--repeats 5]
    python tools/bench_precision.py --profile 3      # torch.profiler kernel table of a few precision-3 learn calls (separate run)

Timing: one DDPGPopulation with seeded weights and inputs; every learn call computes gradients only (apply_updates=False), so each
call does the same work.  After a warm-up of every precision, each repeat times `--calls` back-to-back calls per precision with CUDA
events, the precisions alternating inside the repeat; the median over repeats is reported.  The inputs and activations (GBs) are
far larger than the 126 MB L2, so nothing is served warm from it between calls.
Accuracy: the worst per-tensor max-norm error (max |got - oracle| / max |oracle|, the metric of the precision-0 parity tests) of
every gradient tensor of every agent against oracle/ddpg_np.py (fp32 NumPy) at the same batch, and the relative loss errors; and
the same error against a float64 evaluation of the learn step (tools/precision_model.py, no operand rounded), for every precision
and for the fp32 oracle itself, which separates the oracle's own rounding at this batch size from that of the GPU path.
The device name and its power limit are printed with the numbers and stored in the JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import ddpg_np as D  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
import precision_model  # noqa: E402

PRECISIONS = (0, 2, 3)


def seeded_population(A, R, seed=11):
    from avddpg_b200.config import Config
    from avddpg_b200.trainer import DDPGPopulation
    conf = Config(pl_size=A)
    pop = DDPGPopulation(1, A, conf, rows_per_agent=R, precision=0)
    rng = np.random.default_rng(seed)
    nets = []
    for a in range(A):
        four = [D.init_actor(rng), D.init_critic(rng), D.init_actor(rng), D.init_critic(rng)]
        for p in (four[0], four[2]):
            D.randomize_bn(p, rng, [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
        for p in (four[1], four[3]):
            D.randomize_bn(p, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")])
        four[0]["W3"] *= 50; four[1]["W3"] *= 300; four[2]["W3"] *= 50; four[3]["W3"] *= 300
        for bank, net in zip((pop.actor, pop.critic, pop.t_actor, pop.t_critic), four):
            bank.load_named(a, net)
        nets.append(four)
    n = A * R
    s = rng.normal(0, 2, (n, 4)).astype(np.float32)
    act = rng.uniform(-2.5, 2.5, n).astype(np.float32)
    r = -rng.uniform(0, 0.5, n).astype(np.float32)
    s2 = (s + rng.normal(0, 0.2, (n, 4))).astype(np.float32)
    batch = tuple(torch.as_tensor(x, device="cuda").contiguous() for x in (s, act, r, s2))
    return conf, pop, nets, (s, act, r, s2), batch


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unknown ({e})"
    return name, q


def oracle_refs(conf, nets, host, R):
    s, act, r, s2 = host
    refs = []
    for i, (ac, cr, ta, tc) in enumerate(nets):
        rows = slice(i * R, (i + 1) * R)
        batch = (s[rows], act[rows].reshape(-1, 1), r[rows].reshape(-1, 1), s2[rows])
        refs.append(D.learn(ac, cr, ta, tc, batch, gamma=conf.gamma, high=conf.action_high))
    return refs


def f64_refs(conf, nets, host, R):
    """float64 gradients of the same learn step (precision_model.emulate with no rounding site): [(critic, actor)] per agent"""
    s, act, r, s2 = host
    return [precision_model.emulate(four, (s[i * R:(i + 1) * R], act[i * R:(i + 1) * R], r[i * R:(i + 1) * R], s2[i * R:(i + 1) * R]), {},
                                    gamma=conf.gamma, high=conf.action_high) for i, four in enumerate(nets)]


def worst_error(grads, refs):
    """grads(i, kind, name) -> array; refs: [(critic dict, actor dict)] -> (worst max-norm error, where)"""
    worst, where = 0.0, None
    for i, (rc, ra) in enumerate(refs):
        for kind, ref in (("critic", rc), ("actor", ra)):
            for name, want in ref.items():
                got = np.asarray(grads(i, kind, name), np.float64)
                want = np.asarray(want, np.float64).reshape(got.shape)
                e = float(np.max(np.abs(got - want)) / max(np.max(np.abs(want)), 1e-300))
                if e > worst:
                    worst, where = e, f"agent {i} {kind}.{name}"
    return worst, where


def errors(pop, refs, refs64):
    bank = {"critic": pop.critic, "actor": pop.actor}
    got = lambda i, kind, name: bank[kind].view(name, i, bank[kind].grad).cpu().numpy()
    worst, where = worst_error(got, [(ocg, oag) for ocg, oag, _ in refs])
    worst64, where64 = worst_error(got, refs64)
    loss_err = 0.0
    for i, (_, _, info) in enumerate(refs):
        loss = pop.loss[i].cpu().numpy().astype(np.float64)
        for k, key in enumerate(("critic_loss", "actor_loss")):
            loss_err = max(loss_err, abs(loss[k] - info[key]) / max(1.0, abs(info[key])))
    return worst, where, worst64, where64, loss_err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=4)
    ap.add_argument("--rows", type=int, default=262_144)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_precision3.json"))
    ap.add_argument("--profile", type=int, default=None, metavar="PRECISION", help="torch.profiler kernel table instead of the timing")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_precision.py needs a CUDA device")
    A, R = args.agents, args.rows
    conf, pop, nets, host, (s, act, r, s2) = seeded_population(A, R)
    name, power = device_info()
    print(f"device: {name}; power limit, max SM clock: {power}", flush=True)

    def call(prec):
        pop.precision = prec
        pop.learn(s, act, r, s2, apply_updates=False)

    if args.profile is not None:
        from torch.profiler import ProfilerActivity, profile
        for _ in range(3):
            call(args.profile)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                call(args.profile)
            torch.cuda.synchronize()
        print(f"precision {args.profile}, {A} x {R} rows, 5 learn calls")
        print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25))
        return

    result = {"what": "learn call (gradients only) at the C2 learn shape, CUDA events, median of repeats", "device": name,
              "power_limit_and_max_sm_clock": power, "agents": A, "rows_per_agent": R, "calls_per_repeat": args.calls,
              "repeats": args.repeats, "precisions": {}}
    refs = oracle_refs(conf, nets, host, R)
    refs64 = f64_refs(conf, nets, host, R)
    o64, o64_where = worst_error(lambda i, kind, name: refs[i][0 if kind == "critic" else 1][name], refs64)
    result["fp32_oracle_vs_float64"] = {"worst_tensor_max_norm_error": o64, "worst_tensor": o64_where}
    print(f"fp32 oracle (oracle/ddpg_np.py) vs float64: worst per-tensor error {o64:.2e} ({o64_where})", flush=True)
    for prec in PRECISIONS:               # accuracy first: one call per precision on the seeded weights
        call(prec)
        torch.cuda.synchronize()
        worst, where, worst64, where64, loss_err = errors(pop, refs, refs64)
        result["precisions"][str(prec)] = {"worst_tensor_max_norm_error": worst, "worst_tensor": where,
                                           "worst_tensor_max_norm_error_vs_float64": worst64, "worst_tensor_vs_float64": where64,
                                           "worst_loss_error": loss_err}
        print(f"precision {prec}: worst per-tensor error {worst:.2e} ({where}) against the fp32 oracle, {worst64:.2e} ({where64}) "
              f"against float64; losses {loss_err:.2e}", flush=True)
    for prec in PRECISIONS:               # warm-up of every shape and workspace
        for _ in range(3):
            call(prec)
    torch.cuda.synchronize()
    times = {p: [] for p in PRECISIONS}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for rep in range(args.repeats):
        for prec in (PRECISIONS if rep % 2 == 0 else PRECISIONS[::-1]):
            call(prec)                    # the first call after a switch of precision is not timed
            ev[0].record()
            for _ in range(args.calls):
                call(prec)
            ev[1].record()
            torch.cuda.synchronize()
            times[prec].append(ev[0].elapsed_time(ev[1]) / args.calls)
    for prec in PRECISIONS:
        med = statistics.median(times[prec])
        result["precisions"][str(prec)].update(learn_ms_median=med, learn_ms_all=times[prec])
        print(f"precision {prec}: learn {med:.3f} ms (median of {args.repeats}; {', '.join(f'{t:.3f}' for t in times[prec])})")
    result["speedup_3_over_0"] = result["precisions"]["0"]["learn_ms_median"] / result["precisions"]["3"]["learn_ms_median"]
    print(f"precision 3 is {result['speedup_3_over_0']:.2f}x faster than precision 0")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
