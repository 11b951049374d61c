#!/usr/bin/env python
"""bench.py -- avddpg hot path on B200: platoon env-steps/s (+ DDPG updates/s) vs the reference CPU path.

    python bench.py --gpus N --steps K --warmup W            # native arm (this repo's CUDA path), config c2
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: CPU port of the reference loop
    python bench.py --config {c1,c2,c3,c4,sweep} ...         # the other BASELINE.json configs (same JSON contract)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one pass of the hot path over the population of the chosen config on each GPU:
act (actor forward) -> OU noise + clip -> Platoon.step -> ReplayBuffer.add for every agent -> replay sample (64 per ring) ->
DDPG learn -> federated round (interfrl, gradients, every step: local reduce -> ONE NVLink kernel that reduces in the switch and
applies Adam + Polyak) -- the exchange is INSIDE the timed step on every GPU count.

  c1  BASELINE configs[0]: 1 platoon x 2 followers, no FRL (the reference's default `python run.py tr`)
  c2  BASELINE configs[1]: 4096 platoons x 4 followers per GPU (the N=1 headline; default)
  c3  BASELINE configs[2]: 8 platoons x 4 followers, FedAvg of actor/critic gradients every step
  c4  BASELINE configs[3]: 65,536 platoons x 8 followers over 8 GPUs = 8192 x 8 per GPU, NVLS allreduce aggregation every step
  sweep  BASELINE configs[4]: env-step kernel, 2^10 .. 2^24 platoons, M in {4, 8}, plain and training launch, vs the HBM roofline

Weak scaling: every rank owns its own platoons (global platoon ids are offset by rank, so RNG streams do not depend on the GPU
count); the only data-path collective is the FRL exchange.  Every config replays the training step as a captured CUDA graph
(`BatchedTrainer.capture / replay`; the FRL epoch and buffer half live in device memory, so the NVLink exchange replays too);
`--eager` launches it kernel by kernel (C2: 1.094 vs 1.072 ms per step).

The JSON line also carries
  roofline     : the dominant kernel group (learn step: tensor pipe) + roofline_env / roofline_env_train (HBM), CUDA-event timed
  e2e          : the same step driven through host buffers (pinned H2D of the leader inputs, D2H of the per-step reward/done
                 statistics and losses) every step;  e2e_env_host: Platoon.step through HOST buffers (actions in, obs/reward/done out)
  precision0   : the same step with the fp32 SIMT parity kernels (precision = 0)
  cpu_baseline : oracle port of the reference loop on this box's host cores (rank 0, N=1 only)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "platoon-vehicle env-steps/s"
RING_CAP, BATCH = 100_000, 64
CONFIGS = {
    # G platoon-groups per GPU (agents of a group share nothing; groups of one follower index are the FRL system), E envs per group
    "c1": dict(G=1, E=1, M=2, fed=False, graph=True,
               workload="C1: 1 platoon x 2 followers (reference default run), decentralized Model B euler, OU noise, replay cap 100000, batch 64"),
    "c2": dict(G=1, E=4096, M=4, fed=True, graph=True,
               workload="C2: 4096 platoons x 4 followers per GPU, decentralized Model B euler, OU noise, replay cap 100000, batch 64"),
    "c3": dict(G=8, E=1, M=4, fed=True, graph=True,
               workload="C3: 8 platoons x 4 followers, interfrl FedAvg of actor/critic gradients every step, replay cap 100000, batch 64"),
    "c4": dict(G=1, E=8192, M=8, fed=True, graph=True,
               workload="C4: 8192 platoons x 8 followers per GPU (65,536 x 8 on 8 GPUs), interfrl allreduce aggregation every step, batch 64"),
}


def _ncu_traffic():
    """DRAM bytes per launch from the committed `ncu --set full` captures (profiles/r02_traffic.json, written by tools/ncu_traffic.py
    from the captures named in its "source" key; falls back to the round-1 file): {"env": bytes per env_step_kernel launch at the
    roofline population, "learn": bytes summed over the launches of one learn step at C2}."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        d = json.load(open(path))
        env = next((v for k, v in d.items() if "env" in k and isinstance(v, list)), [])
        learn = next((v for k, v in d.items() if "learn" in k and isinstance(v, list)), [])
        tot = lambda rows: float(sum(r["dram_read_bytes"] + r["dram_write_bytes"] for r in rows)) if rows else None
        return {"env": tot(env[:1]), "learn": tot(learn), "file": f"profiles/{name}"}
    return {"env": None, "learn": None, "file": None}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d.get("bf16_tflops", 1590.0)),
                    tf_sustained=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1590.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(float(os.environ.get("AVD_CLOCK_PERIOD", "0.05")))

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = int(float(self.rows[0][1])) if self.rows else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _dist_setup():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def _max_over_ranks(ms, world):
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _timed(fn, n, world):
    import torch
    _barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    _barrier(world)
    return _max_over_ranks(e0.elapsed_time(e1), world) / n


# --------------------------------------------------------------------------------------------- native arm
LEARN_MACS_PER_SAMPLE = 340_464          # SURVEY.md §8d: reference-equivalent MACs per sampled transition
ENV_BYTES_PER_VEHICLE_STEP = 48          # SURVEY.md §8d: x[4], prev_a, u in; x'[4], prev_a', reward out
ENV_TRAIN_BYTES_PER_VEHICLE_STEP = 112   # + OU state r/w and applied action (16) + replay record (40) + episodic reward r/w (8); + 8/M episode counters


def build_trainer(cfg, rank, world, precision, pg, ring_cap=None):
    import torch
    from avddpg_b200.config import Config
    from avddpg_b200.trainer import BatchedTrainer
    G, E, M = cfg["G"], cfg["E"], cfg["M"]
    if cfg is CONFIGS["c3"] and world > 1:              # 8 platoons in total: shard them
        G = max(1, G // world)
    kw = dict(pl_size=M, num_platoons=G * E)
    if cfg["fed"]:
        # interfrl / gradients / every step; plain mean: the |1/mean reward| weights only start after weighted_window full episodes
        # (trainer.py:640-641: 10 x 600 steps), far beyond a benchmark run, and are covered by tests/test_gpu_ddpg.py
        kw.update(fed_method="interfrl", weighted_average_enabled=False)
    conf = Config(**kw)
    # sized from the device's total memory, not from what happens to be free, so that the same arguments give the same ring (and the
    # same sampled inputs) on every run; a ring above half of the device's memory is shrunk to 35 % of it (the JSON line reports it)
    total = torch.cuda.get_device_properties(torch.cuda.current_device()).total_memory
    cap = RING_CAP if ring_cap is None else ring_cap
    per_slot = M * G * E * 40
    if cap * per_slot > 0.5 * total:
        cap = int(0.35 * total / per_slot)
    free, _ = torch.cuda.mem_get_info()
    if cap * per_slot > free:
        raise RuntimeError(f"the {cap}-slot replay ring needs {cap * per_slot / 1e9:.1f} GB, but only {free / 1e9:.1f} GB of device memory "
                           "are free (the ring is sized for a device the benchmark has to itself)")
    tr = BatchedTrainer(conf, num_groups=G, envs_per_group=E, ring_capacity=cap, rank=rank, world=world,
                        process_group=pg if cfg["fed"] else None, precision=precision)
    if E >= 64:
        tr.rings.fill_synthetic()        # steady state: sampling range == capacity from the first timed step
        tr.buffer_counter = cap
    else:
        for _ in range(conf.batch_size + 8):
            tr.step()
    return conf, tr


def time_env_roofline(P_big, M, train, steps=30, warmup=5):
    """Env-step kernel alone on a population whose working set exceeds L2 (126 MB): CUDA events around each launch on the launching
    stream, average duration -> achieved algorithmic GB/s.  train=False: actions and leader inputs supplied (48 B per vehicle-step
    + 5 B per platoon); train=True: the launch the training loop makes (OU + clip + leader draw + replay record + episodic bookkeeping:
    112 B per vehicle-step + 8 B per platoon)."""
    import torch
    from avddpg_b200.config import Config
    from avddpg_b200.environment import BatchedPlatoons
    from avddpg_b200.replaybuffer import ReplayRings
    if train:
        conf = Config(pl_size=M)
        rings = ReplayRings(4, M, P_big, 64)
        env = BatchedPlatoons(P_big, M, conf, ring=rings, clock=rings.clock, auto_reset=True, track_kinematics=False)
        step = lambda: env.step_native(explore=True, gen_exog=True, advance_clock=True)
        alg = P_big * (M * ENV_TRAIN_BYTES_PER_VEHICLE_STEP + 8.0)
    else:
        conf = Config(pl_size=M, can_terminate=False)
        env = BatchedPlatoons(P_big, M, conf, track_kinematics=False, track_episodes=False, store_actions=False)
        step = lambda: env.step_native(leader_exog=True, advance_clock=False)
        alg = P_big * (M * ENV_BYTES_PER_VEHICLE_STEP + 5.0)
    env.reset()
    env.action_mu.normal_(0, 0.5)
    env.leader_exog.normal_(0, 0.1)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in evs)
    avg = sum(ms) / len(ms)
    del env
    torch.cuda.empty_cache()
    return dict(avg_ms=avg, min_ms=ms[0], alg_bytes=alg, working_set_mb=P_big * M * 4 * 11 / 1e6)


def env_host_leg(M, P, steps):
    """Platoon.step through HOST buffers -- the call a host-driven consumer of the reference's Platoon.step makes
    (avd_env_step_host: actions [M][P] + leader inputs [P] in, obs [4][M][P] + reward [M][P] + done [P] out, synchronous)."""
    import ctypes as C
    import torch
    from avddpg_b200 import _lib
    from avddpg_b200.config import Config
    from avddpg_b200.environment import BatchedPlatoons
    conf = Config(pl_size=M)
    env = BatchedPlatoons(P, M, conf, track_kinematics=False)
    env.reset()
    pin = lambda *shape, dt=torch.float32: torch.zeros(*shape, dtype=dt).pin_memory()
    act, exog, obs, rew, done = pin(M, P), pin(P), pin(4, M, P), pin(M, P), pin(P, dt=torch.uint8)
    act.normal_(0, 0.5)
    exog.normal_(0, 0.1)
    lib = _lib.load()

    def one():
        env._prepare(False, False, True, False)
        _lib.check(lib.avd_env_step_host(C.byref(env.prm), C.byref(env.io), C.c_void_p(act.data_ptr()), C.c_void_p(exog.data_ptr()),
                                         C.c_void_p(obs.data_ptr()), C.c_void_p(rew.data_ptr()), C.c_void_p(done.data_ptr()), _lib.current_stream()))
        env._cur ^= 1

    for _ in range(3):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / steps
    return {"value": P * M / dt, "unit": METRIC, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": (M * P + P) * 4,
            "d2h_bytes_per_step": (4 * M * P + M * P) * 4 + P, "api": "avd_env_step_host (synchronous: H2D actions + leader inputs, kernel, D2H obs + "
            "reward + done, stream sync) on pinned host buffers"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(tr, out_dir):
    """Write what the last training step handed its caller to out_dir/<name>.npy (float32): the observations, rewards and done flags
    of every platoon, the applied (OU-perturbed, clipped) actions, the learn losses and local gradients, and the weights of the four
    networks of every agent.  Two builds run with the same arguments see the same inputs, so their files compare one to one."""
    import numpy as np
    env, pop = tr.env, tr.pop
    arrays = {"obs": env.obs, "reward": env.reward, "done": env.done, "action": env.action_out.t(), "loss": pop.loss,
              "actor_grad": pop.actor.grad, "critic_grad": pop.critic.grad, "actor": pop.actor.flat, "critic": pop.critic.flat,
              "target_actor": pop.t_actor.flat, "target_critic": pop.t_critic.flat}
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total / 2**20:.1f} MB of outputs exceed the {DUMP_LIMIT_BYTES >> 20} MB limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_native(args):
    import torch
    rank, world, local = _dist_setup()
    from avddpg_b200 import _lib
    _lib.require_device()
    if args.config == "sweep":
        return run_sweep(args, rank, world, local)
    cfg = CONFIGS[args.config]
    pk = _peaks()
    pg = None
    if world > 1:
        import torch.distributed as dist
        pg = dist.group.WORLD
    conf, tr = build_trainer(cfg, rank, world, args.precision, pg)
    env, rings, pop = tr.env, tr.rings, tr.pop
    P, M = env.P, env.M
    warm = max(3, args.warmup)
    for _ in range(warm):
        tr.step()
    # The training step is replayed as a captured CUDA graph (BatchedTrainer.capture / replay: two steps per replay, ping-pong state)
    # whenever the FRL transport can be captured (device-resident epoch: local and NVLink peer transports; not NCCL); --eager opts out.
    graph = (cfg["graph"] or args.graph) and not args.eager and (tr.fed is None or tr.fed.graph_safe)
    if graph:
        tr.capture(warmup=1)
    K = args.steps

    def run_steps():                 # EXACTLY K steps: K // 2 replays (+ one eager step when K is odd)
        if graph:
            for _ in range(K // 2):
                tr.replay()
            if K & 1:
                tr.step()
        else:
            for _ in range(K):
                tr.step()

    # ---- device-resident timing of the whole training step (inputs already in HBM; the FRL exchange is part of the step)
    lib = _lib.load()
    l0 = lib.avd_kernel_launches()      # counted inside the library, one per kernel launch site executed
    clk = ClockSampler(local)           # nvidia-smi takes ~0.1 s per query: keep sampling through all timed legs
    clk.__enter__()
    ms_step = _timed(run_steps, 1, world) / K
    launches = lib.avd_kernel_launches() - l0
    if graph:      # replays do not pass through the launch sites: kernels per captured step x replayed steps (+ the eager one)
        launches += (K // 2) * 2 * tr.kernels_per_step
    value = world * P * M / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:      # before the legs below move the state on
        dump_outputs(tr, args.dump_outputs)

    # ---- attribution: env part (act + env step + replay add), learn part (sample + learn), FRL round (reduce + fused consumer)
    def env_part():
        pop.act(env.native_state, env.action_mu, tr.E)
        env.step_native(explore=True, gen_exog=True, advance_clock=False)
        rings.clock.advance(step=1, ring=1)

    def learn_part():
        s, a, r, s2 = rings.sample(advance_clock=True)
        pop.learn(s, a, r, s2, apply_updates=tr.fed is None)

    n_attr = max(30, min(60, args.steps))
    ms_env = _timed(env_part, n_attr, world)
    ms_learn = _timed(learn_part, n_attr, world)
    # the tensor-core roofline is quoted on the learn call ALONE (its 15 launches; the HBM-bound replay gather of learn_part is a different
    # kernel): one sampled batch reused -- the step streams ~2 GB of backward tiles through DRAM, 16 x the 126 MB L2, between two uses
    batch = rings.sample(advance_clock=True)
    # A BURST measurement, to be read against the burst peak: by now the GPU has run ~0.2 s of back-to-back steps and sits at its power
    # cap (`clocks.reasons`), where the same call takes ~5 % longer (tools/profile_learn.py: 0.948 ms for 20-50 calls, 0.997 for 100, 1.028
    # for 300).  So: one second of idle, then 30 calls; the figure of the loaded state is kept beside it and read against the SUSTAINED peak.
    ms_learn_loaded = _timed(lambda: pop.learn(*batch, apply_updates=tr.fed is None), n_attr, world)
    torch.cuda.synchronize()
    time.sleep(1.0)
    ms_learn_only = _timed(lambda: pop.learn(*batch, apply_updates=tr.fed is None), 30, world)
    frl = None
    if tr.fed is not None:
        ms_frl = _timed(lambda: tr.fed.aggregate_gradients(write_back=False), 50, world)
        frl = {"mode": "interfrl / gradients / unweighted, every step", "round_us": ms_frl * 1e3, "in_timed_step": True,
               "payload_bytes": int(M * (pop.actor.n_train + pop.critic.n_train + 1) * 4), "ranks": world, "transport": tr.fed.transport,
               "launches_per_round": 2,
               "collective": ("avd_fed_reduce2 -> fed_apply_kernel: cross-rank barrier, multimem.ld_reduce over the NVLS multicast mapping "
                              "(in-switch reduction), division, Adam x2, Polyak x2, step counters in ONE kernel (csrc/avd_peer.cu)"
                              if world > 1 else "avd_fed_reduce2 -> fed_apply_kernel (single rank: no exchange; same fused consumer)")}
        if world > 1 and not args.quick:    # the NCCL transport (all_reduce + finalize + broadcast + Adam/Polyak) for comparison
            from avddpg_b200.server.federated import FederatedAggregator
            agg_nccl = FederatedAggregator(pop, conf, process_group=pg, transport="nccl")
            for _ in range(5):
                agg_nccl.aggregate_gradients()
            frl["round_us_nccl_transport"] = _timed(lambda: agg_nccl.aggregate_gradients(), 50, world) * 1e3

    # ---- end to end through host buffers: pinned leader inputs in, reward/done statistics + losses out, every step.
    # HostStepPipeline double-buffers both directions, so the host reads the results of step k - 1 while step k runs.
    from avddpg_b200.trainer import HostStepPipeline
    pipe = HostStepPipeline(tr)
    gen = torch.Generator().manual_seed(1 + rank)
    acc = 0.0

    def e2e_step():
        pipe.input_buffer().normal_(0, 0.1, generator=gen)
        prev = pipe.submit()
        return float(prev[0]) if prev is not None else 0.0

    for _ in range(3):
        e2e_step()
    pipe.drain()
    _barrier(world)
    n_e2e = max(5, min(args.steps, 50))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        acc += e2e_step()
    acc += float(pipe.drain()[0])                    # the last step's results: the timed region ends with the GPU drained
    _barrier(world)
    e2e_ms = _max_over_ranks((time.perf_counter() - t0) * 1e3, world) / n_e2e
    e2e = {"value": world * P * M / (e2e_ms * 1e-3), "unit": METRIC, "h2d_bytes_per_step": pipe.h2d_bytes_per_step,
           "d2h_bytes_per_step": pipe.d2h_bytes_per_step, "ms_per_step": e2e_ms, "steps": n_e2e,
           "api": "HostStepPipeline(BatchedTrainer).submit(): pinned H2D of the leader inputs + eager step + D2H of reward/done "
                  "statistics and losses every step; results are read on the host one step behind (double-buffered pinned buffers)"}
    clk.__exit__(None, None, None)

    # ---- the fp32 SIMT parity kernels (precision = 0) on the same step, beside the tensor-core number
    p0 = None
    if args.precision != 0 and not args.quick:
        saved = pop.precision
        pop.precision = 0
        tr.step()
        ms_p0 = _timed(lambda: tr.step(), 3, world)
        pop.precision = saved
        p0 = {"ms_per_step": ms_p0, "value": world * P * M / (ms_p0 * 1e-3), "unit": METRIC, "steps": 3,
              "what": "the same training step with precision = 0 (fp32 SIMT learn kernels, 2e-4 parity against the oracle)"}

    out = None
    if rank == 0:
        rows = pop.A * pop.R
        learn_flops = 2.0 * LEARN_MACS_PER_SAMPLE * rows
        learn_tf = learn_flops / (ms_learn_only * 1e-3) / 1e12
        traffic = _ncu_traffic()
        # the learn leg is ~n_attr x 1 ms of back-to-back tensor work: a burst measurement -> burst peak; the sustained figure is given too
        op = {0: "fp32 SIMT parity kernels", 1: "bf16", 2: "fp16"}[args.precision]
        roofline_learn = {"bound": "tensor", "kernel": (f"learn step: 6 fused pass launches (fused3_kernel) + 2 wgrad3 + 2 dgrad3, {op} tcgen05"
                                                       if args.precision else "learn step, fp32 SIMT parity mode"),
                          "achieved": learn_tf, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": learn_tf / pk["tf_burst"],
                          "frac_of_sustained_peak": learn_tf / pk["tf_sustained"], "peak_sustained": pk["tf_sustained"],
                          "traffic": traffic["learn"] if (args.precision and args.config == "c2") else None,
                          "traffic_unit": f"DRAM bytes per learn step, summed over its launches (ncu --set full, {traffic['file']})",
                          "peak_source": pk["src"] + ": cuBLAS bf16 burst (the leg is a few ms of back-to-back launches); fp16 and bf16 share the rate",
                          "alg_flops_per_step": learn_flops, "alg_macs_per_sample": LEARN_MACS_PER_SAMPLE, "rows_per_step": rows,
                          "learn_ms": ms_learn_only, "timed_iterations": 30, "regime": "burst: 30 back-to-back learn calls after 1 s of idle",
                          "learn_ms_under_power_cap": ms_learn_loaded,
                          "frac_of_sustained_peak_under_power_cap": learn_flops / (ms_learn_loaded * 1e-3) / 1e12 / pk["tf_sustained"],
                          "learn_ms_with_replay_sample": ms_learn,
                          "l2": "inputs (42 MB at C2) are reused, but every step streams ~2 GB of backward tiles through DRAM (16 x the L2) in between"}
        roofline_env = roofline_env_train = None
        if not args.quick:
            big = args.roofline_platoons if M <= 4 else args.roofline_platoons // 2
            for train in (False, True):
                rl = time_env_roofline(big, M, train)
                achieved = rl["alg_bytes"] / (rl["avg_ms"] * 1e-3) / 1e9
                d = {"bound": "hbm", "kernel": f"env_step_kernel<{M}>" + (" (training launch: OU + clip + leader draw + replay record + "
                                                                         "episodic bookkeeping fused)" if train else " (actions supplied)"),
                     "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"],
                     "traffic": traffic["env"] if (not train and big == 4 * 1024 * 1024 and M == 4) else None,
                     "traffic_unit": f"DRAM bytes per launch (ncu --set full, {traffic['file']})", "alg_bytes_per_launch": rl["alg_bytes"],
                     "peak_source": pk["src"], "population": f"{big} platoons x {M} (working set {rl['working_set_mb']:.0f} MB > 126 MB L2)",
                     "alg_bytes_per_vehicle_step": ENV_TRAIN_BYTES_PER_VEHICLE_STEP + 8.0 / M if train else ENV_BYTES_PER_VEHICLE_STEP,
                     "avg_launch_ms": rl["avg_ms"], "vehicle_steps_per_s": big * M / (rl["avg_ms"] * 1e-3)}
                if train:
                    roofline_env_train = d
                else:
                    roofline_env = d
        dominant = roofline_learn if (ms_learn > ms_env or roofline_env_train is None) else roofline_env_train
        env_host = None if args.quick else env_host_leg(M, P, 30)
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not args.quick:
            from oracle import cpu_baseline
            cpu = cpu_baseline.time_env_steps(M=M, target_seconds=args.cpu_seconds, with_learn=True)
            cpu_env = cpu_baseline.time_env_steps(M=M, target_seconds=max(2.0, args.cpu_seconds / 3), with_learn=False)
            cpu["env_only_loop"] = {"value": cpu_env["value"], "sample": cpu_env["sample"]}
        agent_updates = world * pop.A / (ms_step * 1e-3)
        out = {"metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": K, "warmup": warm,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": {0: "f32", 1: "bf16", 2: "fp16"}[args.precision], "data": "synthetic", "impl": "native",
               "config": {"workload": cfg["workload"]},
               "details": {"config": args.config, "platoons_per_gpu": P, "followers": M, "agents_per_gpu": pop.A, "rows_per_agent_update": pop.R,
                           "ring_capacity": rings.capacity, "cuda_graph": bool(graph),
                           "l2": f"replay gathers hit a pre-filled {rings.capacity * M * P * 40 / 1e9:.1f} GB ring and the learn workspace is "
                                 f"{(pop._ws.numel() if pop._ws is not None else 0) / 1e9:.1f} GB (both >> 126 MB L2 at c2 / c4); "
                                 "env rooflines measured on > L2 populations",
                           "step": "act(actor fwd) + OU/clip + Platoon.step + ReplayBuffer.add + sample(64/ring) + learn + "
                                   + ("federated round (reduce + fused exchange/Adam/Polyak)" if tr.fed is not None else "Adam x2 + Polyak x2"),
                           "learn_operands": op + (" (fp32 accumulation in TMEM; layer 1 hi/lo-split bf16; heads, losses, Adam, Polyak fp32)" if args.precision else "")},
               "clocks": clk.summary(), "e2e": e2e, "e2e_env_host": env_host, "gpu_launches": launches,
               "roofline": dominant, "roofline_env": roofline_env, "roofline_env_train": roofline_env_train, "roofline_learn": roofline_learn,
               "cpu_baseline": cpu, "precision0": p0,
               "platoon_steps_per_s": value / M,
               # one reference update = learn + Adam x2 + Polyak for ONE (platoon, follower) minibatch of 64 (SURVEY 8d): the step
               # processes platoons x followers of them per GPU; with weight sharing across a group's platoons (DESIGN 9) they are
               # applied as ONE Adam/Polyak step per agent on the mean gradient -- both counts are given
               "ddpg_minibatch_gradients_per_s": world * P * M / (ms_step * 1e-3),
               "ddpg_weight_updates_per_s": agent_updates,
               "ms_env_part": ms_env, "ms_learn_part": ms_learn, "frl": frl}
        print(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return out


def run_sweep(args, rank, world, local):
    """BASELINE configs[4]: env-step kernel over 2^10 .. 2^24 platoons, M in {4, 8}; every rank sweeps its own shard (weak), the
    per-point value is the sum over ranks at the max-over-ranks time.  The JSON line's `value` is the best training-launch point."""
    import torch
    pk = _peaks()
    pts = []
    clk = ClockSampler(local)
    clk.__enter__()
    for M in (4, 8):
        for e in range(10, 25):
            P = 1 << e
            if P * M > (1 << 26):
                continue
            for train in (False, True):
                if train and P * M > (1 << 25):      # 4-slot ring = 160 B per vehicle: keep the sweep far from the HBM capacity
                    continue
                rl = time_env_roofline(P, M, train, steps=args.steps, warmup=max(3, args.warmup))
                ms = _max_over_ranks(rl["avg_ms"], world)
                gbs = rl["alg_bytes"] / (ms * 1e-3) / 1e9
                pts.append({"platoons_per_gpu": P, "followers": M, "mode": "train" if train else "plain", "us": ms * 1e3,
                            "vehicle_steps_per_s": world * P * M / (ms * 1e-3), "alg_GBps_per_gpu": gbs, "frac_of_hbm": gbs / pk["hbm"]})
    clk.__exit__(None, None, None)
    if rank == 0:
        best = max((p for p in pts if p["mode"] == "train"), key=lambda p: p["vehicle_steps_per_s"])
        bestp = max((p for p in pts if p["mode"] == "plain"), key=lambda p: p["vehicle_steps_per_s"])
        print(json.dumps({"metric": METRIC, "value": best["vehicle_steps_per_s"], "unit": METRIC, "n_gpus": world, "steps": args.steps,
                          "warmup": max(3, args.warmup), "ms_per_step": best["us"] * 1e-3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "native",
                          "config": {"workload": "sweep: env-step kernel, 2^10..2^24 platoons x {4, 8} followers per GPU, plain (48 B/vehicle-step) "
                                                 "and training launch (112 B/vehicle-step) vs the HBM roofline"},
                          "clocks": clk.summary(), "gpu_launches": len(pts) * (args.steps + max(3, args.warmup)),
                          "roofline": {"bound": "hbm", "kernel": "env_step_kernel (training launch, best point)", "achieved": best["alg_GBps_per_gpu"],
                                       "peak": pk["hbm"], "unit": "GB/s", "frac": best["frac_of_hbm"], "traffic": None, "peak_source": pk["src"]},
                          "best_plain": bestp, "best_train": best, "points": pts, "e2e": None, "cpu_baseline": None}))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """Reference arm: the CPU port of the reference's own loop (oracle/), all host cores, rank 0 only.
    Each bench "step" is a bounded sample: every core steps one platoon of the config's length for ~budget seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline
    cfg = CONFIGS[args.config if args.config in CONFIGS else "c2"]
    total = args.steps
    budget = max(0.25, min(args.cpu_seconds, 150.0 / (total + args.warmup)))
    pool = cpu_baseline.EnvLoopPool(M=cfg["M"], with_learn=True)
    vals, steps, slowest = [], 0, 0.0
    try:
        for i in range(args.warmup + total):
            v, steps, slowest = pool.run(budget)
            if i >= args.warmup:
                vals.append(v)
    finally:
        pool.close()
    v = sum(vals) / len(vals)
    line = {"metric": METRIC, "value": v, "unit": METRIC, "n_gpus": args.gpus, "steps": total, "warmup": args.warmup,
            "ms_per_step": slowest * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference", "config": {"workload": cfg["workload"]},
            "cpu_baseline": {"value": v, "unit": METRIC, "cores": pool.cores, "kind": "port", "sample": pool.describe(steps, slowest)},
            "e2e": {"value": v, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4", "sweep"])
    ap.add_argument("--roofline-platoons", type=int, default=4 * 1024 * 1024)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="main timing, attribution and e2e only (no rooflines, precision-0 or CPU legs)")
    ap.add_argument("--precision", type=int, default=2,
                    help="learn kernels: 0 fp32 SIMT (parity mode), 1 bf16 tcgen05, 2 fp16 tcgen05 (default; DESIGN.md section 4)")
    ap.add_argument("--graph", action="store_true", help="replay a captured CUDA graph of the training step (the default of every config)")
    ap.add_argument("--eager", action="store_true", help="launch the training step kernel by kernel instead of replaying its CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (observations, rewards, done flags, actions, losses, "
                         "gradients, weights) to DIR/<name>.npy (rank 0; configs c1-c4)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == "sweep"):
        ap.error("--dump-outputs needs the native training step (configs c1-c4)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
