"""Seed sweeps as one batch: time the graph-replayed training step of S independently seeded runs (BatchedTrainer seeds=[...]) and
compare it with S separate runs, i.e. S x the step time of one run (what one process per seed costs on a GPU that time-slices them).

    python tools/bench_runs.py [--out profiles/r04_runs.json] [--window 1.0] [--quick]
    python tools/bench_runs.py --sweep [--out profiles/r05_sweep.json] [--window 0.5] [--quick]

Shapes: C1 (one platoon of 2 followers per run) at S in {1, 16, 128, 1024} and C3 (8 platoons of 4 followers, unweighted interfrl,
whose FRL schedule can be captured) at S in {1, 16, 128}; ring 100,000 slots, batch 64, precisions 0 and 2.  S = 1 is the default
trainer without a run table.  Every ring is filled with synthetic transitions first, so each step samples from the full ring
(steady state).  Step times come from CUDA events around back-to-back graph replays (two steps each) over a window of at least
--window seconds, after warm-up replays.  The GPU name, power limit and max SM clock are read with nvidia-smi in the same process.

--sweep: the cost of per-run hyperparameters.  At C1 and C3, S in {16, 128}, precisions 0 and 2, the same batch is built twice --
seeds only, and seeds with overrides whose learning rates, gamma, tau, std_dev and theta differ from run to run (per-agent table in
the learn step, per-run OU parameters in the env step) -- and the two captured graphs are timed alternately, --reps windows each.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = {
    "c1": dict(num_groups=1, pl_size=2, fed_method="normal", runs=(1, 16, 128, 1024)),
    "c3": dict(num_groups=8, pl_size=4, fed_method="interfrl", runs=(1, 16, 128)),
}
RING, BATCH = 100_000, 64


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def _captured(shape: str, S: int, precision: int, ring: int, overrides=None):
    from avddpg_b200.config import Config
    from avddpg_b200.trainer import BatchedTrainer
    sh = SHAPES[shape]
    conf = Config(pl_size=sh["pl_size"], batch_size=BATCH, buffer_size=ring, fed_method=sh["fed_method"], weighted_average_enabled=False)
    seeds = None if S == 1 else list(range(1, S + 1))
    tr = BatchedTrainer(conf, sh["num_groups"], 1, ring_capacity=ring, precision=precision, seeds=seeds, overrides=overrides)
    tr.rings.fill_synthetic()
    tr.buffer_counter = ring
    return tr, tr.capture(warmup=2)


def _replay_ms(graph, n: int) -> float:
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        graph.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def time_point(shape: str, S: int, precision: int, window: float, ring: int):
    import torch
    tr, graph = _captured(shape, S, precision, ring)
    for _ in range(5):
        graph.replay()
    torch.cuda.synchronize()
    n = max(20, math.ceil(window / (_replay_ms(graph, 10) / 10 * 1e-3)))
    ms = _replay_ms(graph, n)
    step_us = ms * 1e3 / (2 * n)
    out = {"shape": shape, "runs": S, "precision": precision, "platoons": tr.P, "agents": tr.pop.A, "kernels_per_step": tr.kernels_per_step,
           "replays": n, "window_s": ms * 1e-3, "step_us": step_us, "run_steps_per_s": S / (step_us * 1e-6)}
    del graph, tr
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def sweep_overrides(S: int):
    """Per-run values around the reference defaults, different from run to run (every key of config.SWEEP_KEYS)."""
    return [dict(actor_lr=5e-5 * (1 + s % 4), critic_lr=5e-4 * (1 + s % 3), gamma=0.99 - 0.01 * (s % 5), tau=1e-3 * (1 + s % 2),
                 std_dev=0.02 * (1 + s % 3), theta=0.15 * (1 + s % 4)) for s in range(S)]


def sweep_point(shape: str, S: int, precision: int, window: float, ring: int, reps: int):
    """The same batch with seeds only and with per-run overrides, each captured; timed in alternating windows."""
    import torch
    variants = {"seeds": _captured(shape, S, precision, ring), "overrides": _captured(shape, S, precision, ring, sweep_overrides(S))}
    for _, graph in variants.values():
        for _ in range(5):
            graph.replay()
    torch.cuda.synchronize()
    n = max(20, math.ceil(window / (_replay_ms(variants["seeds"][1], 10) / 10 * 1e-3)))
    samples = {k: [] for k in variants}
    for _ in range(reps):
        for k, (_, graph) in variants.items():
            samples[k].append(_replay_ms(graph, n) * 1e3 / (2 * n))
    med = {k: sorted(v)[len(v) // 2] for k, v in samples.items()}
    tr = variants["seeds"][0]
    out = {"shape": shape, "runs": S, "precision": precision, "platoons": tr.P, "agents": tr.pop.A, "replays_per_window": n,
           "step_us_seeds": med["seeds"], "step_us_overrides": med["overrides"], "samples_us": samples,
           "overrides_cost": med["overrides"] / med["seeds"] - 1.0,
           "seeds_spread": (max(samples["seeds"]) - min(samples["seeds"])) / med["seeds"]}
    del variants, tr
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON result here as well as to stdout")
    ap.add_argument("--window", type=float, default=1.0, help="seconds of replays per timed point (at least)")
    ap.add_argument("--quick", action="store_true", help="S = 1 and 16 only, ring 1,000 (a check of the tool, not a measurement)")
    ap.add_argument("--sweep", action="store_true", help="time batches with per-run overrides against the same batches with seeds only")
    ap.add_argument("--reps", type=int, default=3, help="--sweep: alternating windows per variant")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_runs.py measures on a CUDA device; none is visible")
    ring = 1000 if args.quick else RING
    info = gpu_info()
    if args.sweep:
        t0 = time.time()
        points = []
        for shape in SHAPES:
            for precision in (0, 2):
                for S in ((16,) if args.quick else (16, 128)):
                    p = sweep_point(shape, S, precision, args.window, ring, args.reps)
                    points.append(p)
                    print(json.dumps(p), flush=True)
        _write({**info, "ring": ring, "batch": BATCH, "window_s": args.window, "reps": args.reps, "wall_s": time.time() - t0,
                "points": points}, args.out)
        return
    t0 = time.time()
    points = []
    for shape, sh in SHAPES.items():
        for precision in (0, 2):
            base = None
            for S in sh["runs"]:
                if args.quick and S > 16:
                    continue
                p = time_point(shape, S, precision, args.window, ring)
                if S == 1:
                    base = p["step_us"]
                p["separate_runs_us"] = S * base
                p["speedup_vs_separate_runs"] = S * base / p["step_us"]
                points.append(p)
                print(json.dumps(p), flush=True)
    res = {**info, "ring": ring, "batch": BATCH, "window_s": args.window, "wall_s": time.time() - t0, "points": points,
           "every_batch_beats_separate_runs": all(p["speedup_vs_separate_runs"] > 1.0 for p in points if p["runs"] > 1)}
    _write(res, args.out)


def _write(res, path):
    line = json.dumps(res)
    print(line)
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
