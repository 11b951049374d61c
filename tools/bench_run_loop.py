"""The per-run episode loop of BatchedTrainer.run (trainers built with seeds) on the device against its host reference loop.

    python tools/bench_run_loop.py [--out profiles/r06_run_loop.json] [--episodes 4] [--reps 5] [--quick]

Shapes: C1 runs (one platoon of 2 followers) at S in {16, 128, 1024}, precision 0; C3 runs (8 platoons of 4 followers, interfrl,
unweighted and weighted with a one-episode window) at S in {16, 128}, precisions 0 and 2.  Episodes are 30 steps long and terminate
early (tight thresholds, small reset states), so the runs end their episodes at different steps.  Every ring is filled with synthetic transitions first,
so every step learns from a full ring.  One trainer per shape runs `run(episodes)` through the device loop (`run()`) and through the
host reference loop (`_run_runs`) in alternating windows, --reps each after one warm-up call of each; a window is a host clock around
one call, which ends synchronised.  Beside them: the graph-replayed `step()` time of the same batch (tools/bench_runs.py: CUDA events
around back-to-back replays of a captured step of a trainer without weighting, whose FRL schedule can be captured), the ceiling
for a loop without episodes.  The GPU name, power limit and max SM clock are read with nvidia-smi in the same process.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_runs import BATCH, SHAPES, _write, gpu_info, time_point  # noqa: E402

RING = 100_000
POINTS = [("c1", "plain", S, 0) for S in (16, 128, 1024)] + \
         [("c3", fed, S, prec) for fed in ("unweighted", "weighted") for prec in (0, 2) for S in (16, 128)]


def _trainer(shape: str, fed: str, S: int, precision: int, ring: int):
    from avddpg_b200.config import Config
    from avddpg_b200.trainer import BatchedTrainer
    sh = SHAPES[shape]
    conf = Config(pl_size=sh["pl_size"], batch_size=BATCH, buffer_size=ring, fed_method=sh["fed_method"], can_terminate=True,
                  reset_ep_max=0.5, reset_max_ev=0.5, max_ep=1.5, max_ev=1.5, episode_sim_time=3.0, weighted_average_enabled=fed == "weighted", weighted_window=1)
    tr = BatchedTrainer(conf, sh["num_groups"], 1, ring_capacity=ring, precision=precision, seeds=list(range(1, S + 1)))
    tr.rings.fill_synthetic()
    tr.buffer_counter = ring
    return tr


def _window(fn, S):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps = fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"s": dt, "steps": steps, "run_steps_per_s": steps * S / dt}


def point(shape, fed, S, precision, episodes, reps, ring, window):
    import torch
    tr = _trainer(shape, fed, S, precision, ring)
    logs = tr.reward_logs()
    loops = {"device": lambda: tr.run(episodes, reward_logs=logs), "host": lambda: tr._run_runs(episodes, logs, True, True)}
    for fn in loops.values():
        fn()                                   # warm-up: builds the device loop's graphs
    samples = {k: [] for k in loops}
    for _ in range(reps):
        for k, fn in loops.items():
            samples[k].append(_window(fn, S))
    rate = {k: sorted(x["run_steps_per_s"] for x in v)[len(v) // 2] for k, v in samples.items()}
    spread = {k: (max(x["run_steps_per_s"] for x in v) - min(x["run_steps_per_s"] for x in v)) / rate[k] for k, v in samples.items()}
    lengths = sorted({n for r in tr.run_episode_steps for n in r})
    out = {"shape": shape, "fed": fed, "runs": S, "precision": precision, "platoons": tr.P, "agents": tr.pop.A, "episodes_per_call": episodes,
           "episode_lengths_seen": lengths, "device_run_steps_per_s": rate["device"], "host_run_steps_per_s": rate["host"],
           "device_over_host": rate["device"] / rate["host"], "spread": spread, "samples": samples}
    del tr, logs, loops
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    ceiling = time_point(shape, S, precision, window, ring)
    out["graph_step_us"] = ceiling["step_us"]
    out["graph_run_steps_per_s"] = ceiling["run_steps_per_s"]
    out["device_share_of_ceiling"] = rate["device"] / ceiling["run_steps_per_s"]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON result here as well as to stdout")
    ap.add_argument("--episodes", type=int, default=4, help="episodes per timed call")
    ap.add_argument("--reps", type=int, default=5, help="alternating windows per loop")
    ap.add_argument("--window", type=float, default=0.5, help="seconds of graph replays for the ceiling")
    ap.add_argument("--quick", action="store_true", help="S = 16 only, ring 1,000 (a check of the tool, not a measurement)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_run_loop.py measures on a CUDA device; none is visible")
    ring = 1000 if args.quick else RING
    info = gpu_info()
    t0 = time.time()
    points = []
    for shape, fed, S, prec in POINTS:
        if args.quick and S != 16:
            continue
        p = point(shape, fed, S, prec, args.episodes, args.reps, ring, args.window)
        points.append(p)
        print(json.dumps({k: v for k, v in p.items() if k != "samples"}), flush=True)
    _write({**info, "ring": ring, "batch": BATCH, "reps": args.reps, "wall_s": time.time() - t0, "points": points,
            "device_never_slower": all(p["device_over_host"] >= 1.0 for p in points)}, args.out)


if __name__ == "__main__":
    main()
