"""Shortest solutions and item queries of the optimal-move query (optimal_moves(ids, pos, paths=True),
K9 ts_optimal_moves).

  python profiles/experiments/optimal_paths.py --out /tmp/optimal_paths.json

65,536 envs of 6x6 / 4 tiles / 8 walls, coloured and single-colour, synthetic() puzzles (mostly
unsolvable) and a solvable() batch in the band [8, 12], at episode start.  Per batch, the commands
below are timed alternately within each repetition (host clock around a call that ends in a device
synchronise; every call reads the free-cell maximum back once), after one warm-up of each:
  query        optimal_moves()                       distance and mask only
  paths        optimal_moves(paths=True)              plus the [254, N] plan
  successors   optimal_moves(ids, pos) on the 4N expand() successors (262,144 items)
  loop         (solvable only) the d-query expert loop: query, step the lowest optimal move, until
               every env has won (max solve_depth queries and steps)
  plan_replay  (solvable only) optimal_moves(paths=True) + playout(actions=plan, record=True)
Reported: median / min / max seconds per command, and checks that the plan replays win in exactly
`distance` moves and that the loop and the plan reach the same final positions.
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

LOWEST_BIT = [0, 0, 1, 0, 2, 0, 1, 0, 3, 0, 1, 0, 2, 0, 1, 0]


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run_batch(ts, env, solvable, reps):
    import torch
    N = env.n_envs
    lowest = torch.tensor(LOWEST_BIT, dtype=torch.uint8, device="cuda")
    succ, _, _ = env.expand()
    s_ids = torch.arange(N, dtype=torch.int32, device="cuda").repeat_interleave(4)
    s_pos = succ.reshape(-1, env.pos_bytes).contiguous()
    names = ("_pos", "_count", "_done", "_flags", "_reward")
    saved = {k: getattr(env, k).clone() for k in names}
    depth = int(env.solve_depth.max()) if solvable else 0

    def restore():
        for k in names:
            getattr(env, k).copy_(saved[k])

    def loop():
        for _ in range(depth):
            _, m = env.optimal_moves()
            env.step(lowest[m.long()])
        return env.pos.clone()

    def plan_replay():
        d, m, plan = env.optimal_moves(paths=True)
        return d, env.playout(actions=plan, record=True)

    cmds = {"query": lambda: env.optimal_moves(), "paths": lambda: env.optimal_moves(paths=True),
            "successors": lambda: env.optimal_moves(s_ids, pos=s_pos)}
    if solvable:
        cmds["loop"] = loop
        cmds["plan_replay"] = plan_replay
    times = {k: [] for k in cmds}
    outs = {}
    for rep in range(reps + 1):                    # repetition 0 is the warm-up
        for k, fn in cmds.items():
            dt, outs[k] = timed(fn)
            if k == "loop":
                restore()
            if rep:
                times[k].append(dt)
    row = {k: dict(seconds_median=statistics.median(v), seconds_min=min(v), seconds_max=max(v)) for k, v in times.items()}
    row["query"]["queries_per_s"] = N / row["query"]["seconds_median"]
    row["paths"]["queries_per_s"] = N / row["paths"]["seconds_median"]
    row["successors"]["queries_per_s"] = 4 * N / row["successors"]["seconds_median"]
    row["paths_over_query"] = row["paths"]["seconds_median"] / row["query"]["seconds_median"]
    d, m = outs["query"]
    d2, m2, _ = outs["paths"]
    row["paths_distance_mask_identical"] = bool(torch.equal(d, d2) and torch.equal(m, m2))
    row["solved_fraction"] = float((d > 0).double().mean())
    if solvable:
        row["loop_over_plan_replay"] = row["loop"]["seconds_median"] / row["plan_replay"]["seconds_median"]
        row["loop_queries"] = depth
        dp, (final, steps, won, _, _) = outs["plan_replay"]
        row["plan_replay_wins_in_distance"] = bool((won == 1).all() and torch.equal(steps, dp))
        row["loop_and_plan_same_final_positions"] = bool(torch.equal(outs["loop"], final))
    return row


def run(args):
    import tiler_slider_b200 as ts
    S, T, W, N = 6, 4, 8, args.envs
    rows = []
    for multi in (True, False):
        for kind in ("synthetic", "solvable_8_12"):
            if kind == "synthetic":
                env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=2024, max_steps=200)
            else:
                env = ts.BatchedTilerSliderEnv.solvable(N, S, T, W, multi, min_depth=8, max_depth=12, seed=2024, max_steps=200)
            row = dict(multi=multi, puzzles=kind, envs=N, **run_batch(ts, env, kind != "synthetic", args.reps))
            rows.append(row)
            print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=7)
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
