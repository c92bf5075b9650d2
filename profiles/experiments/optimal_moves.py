"""Optimal-move query measurements (BatchedTilerSliderEnv.optimal_moves, K9 ts_optimal_moves).

  python profiles/experiments/optimal_moves.py --out /tmp/optimal_moves.json

65,536 envs of 6x6 / 4 tiles / 8 walls, coloured and single-colour: synthetic() puzzles (mostly
unsolvable: the forward search exhausts the reachable set) and a solvable() batch in the band
[8, 12]; each queried at episode start and after 5 and 20 uniformly random steps.  Method of
puzzle_generation.py: one GPU, host clock around a call that ends in a device synchronise (the
call itself reads the free-cell maximum back once), one warm-up call per batch, --reps timed calls.
Reported per case: queries/s (median call), states expanded per query by the forward search and
re-expanded by the backward pass (the kernel's counters), and the distribution of the answers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def measure(env, reps):
    import torch
    env.optimal_moves()                                     # warm-up: plan, scratch slab, module load
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        d, m = env.optimal_moves()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    c = env._optimal.counters.tolist()
    n = env.n_envs
    dist = d.cpu()
    solved = dist[dist > 0].double()
    return dict(envs=n, seconds_median=statistics.median(times), seconds_min=min(times), seconds_max=max(times),
                queries_per_s=n / statistics.median(times),
                forward_states_per_query=c[1] / n, backward_states_per_query=c[2] / n,
                solved_fraction=float((dist > 0).double().mean()), mean_distance_solved=float(solved.mean()) if solved.numel() else None,
                unsolvable=int((dist == -1).sum()), cutoff=int((dist == -2).sum()), not_searched=int((dist == -3).sum()),
                mean_optimal_moves_solved=float(((m.cpu()[dist > 0].unsqueeze(1) >> torch.arange(4, dtype=torch.uint8)) & 1).sum(1).double().mean()) if solved.numel() else None)


def run(args):
    import torch
    import tiler_slider_b200 as ts
    S, T, W, N = 6, 4, 8, args.envs
    rows = []
    for multi in (True, False):
        for kind in ("synthetic", "solvable_8_12"):
            if kind == "synthetic":
                env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=2024, max_steps=200)
            else:
                env = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=8, max_depth=12, seed=2024, max_steps=200)
            gen = torch.Generator(device="cuda").manual_seed(7)
            done_steps = 0
            for steps in (0, 5, 20):
                while done_steps < steps:
                    env.step(torch.randint(0, 4, (N,), dtype=torch.uint8, device="cuda", generator=gen))
                    done_steps += 1
                row = dict(multi=multi, puzzles=kind, random_steps=steps, **measure(env, args.reps))
                rows.append(row)
                print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"card": card(), "shape": "6x6 / 4 tiles / 8 walls", "rows": run(args)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
