"""Hash-table searches (hash_table=True): 5 and 6 tiles, where a state is a 64-bit word, searched by
K11 (optimal_moves) and graded into a band by K7 + K11 (solvable()).

  python profiles/experiments/table_search.py --out /tmp/table_search.json

Workloads, 65,536 envs each at episode start:
  6x6 / 5 tiles / 8 walls, coloured, solvable() [8, 12]
  6x6 / 5 tiles / 8 walls, coloured, synthetic()
  8x8 / 5 tiles / 12 walls, coloured, solvable() [8, 12]
  6x6 / 6 tiles / 8 walls, coloured, solvable() [8, 12]
Every timing is a host clock around a call that ends in a device synchronise; after one warm-up,
`--reps` repetitions, reported as median / min / max.
  generate     solvable(..., hash_table=True): time, rounds, candidates and yield (accepted / candidates)
  k11          optimal_moves(hash_table=True), without and with paths: queries/s; the share of -3
               and the other answers; the plan's table and slab bytes per CTA
  baseline     the first `--baseline` puzzles of the batch through solve_batch (one BfsSolver per
               puzzle, the path it takes for 5 to 8 tiles), timed once, beside K11 on the same puzzles;
               K11's start distance is compared with BfsSolver's solve depth
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


def stats(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def timed(fn, reps):
    """(last result, stats of the host time of fn() over reps runs after one warm-up)."""
    import torch
    out = fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return out, stats(ts)


def run_batch(env, reps, n_baseline):
    import torch
    from tiler_slider_b200.bfs import solve_batch
    n = env.n_envs
    out = {"envs": n}
    (d, m), out["k11_s"] = timed(lambda: env.optimal_moves(hash_table=True), reps)
    out["k11_queries_per_s_median"] = n / out["k11_s"]["median"]
    (dp, mp, _), out["k11_paths_s"] = timed(lambda: env.optimal_moves(paths=True, hash_table=True), reps)
    out["k11_paths_queries_per_s_median"] = n / out["k11_paths_s"]["median"]
    out["k11_paths_equal_no_paths"] = bool(torch.equal(d, dp) and torch.equal(m, mp))
    out["answers"] = {str(k): int((d == k).sum()) for k in (-4, -3, -2, -1)}
    out["answers"][">=1"] = int((d >= 1).sum())
    out["share_not_searched"] = float((d == -3).double().mean())
    out["distance_max"] = int(d.max())
    p = env._optimal._plan_table()
    out["plan"] = {k: p[k] for k in ("grid", "ctas_per_sm", "queue_smem", "table_slots", "spill_per_cta")}
    out["table_bytes_per_cta"] = 8 * p["table_slots"]
    out["slab_bytes_per_cta"] = 8 * p["spill_per_cta"]
    out["counters_fwd_bwd_states"] = env._optimal.counters[1:3].tolist()

    k = min(n_baseline, n)
    sub = type(env).from_puzzles([env.puzzle(i) for i in range(k)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = solve_batch(sub)
    torch.cuda.synchronize()
    t_bfs = time.perf_counter() - t0
    (ds, _), t_k11 = timed(lambda: sub.optimal_moves(hash_table=True), reps)
    out["baseline"] = {"puzzles": k, "solve_batch_s": t_bfs, "solve_batch_puzzles_per_s": k / t_bfs,
                       "k11_same_puzzles_s": t_k11, "k11_same_puzzles_per_s_median": k / t_k11["median"],
                       "k11_speedup_median": t_bfs / t_k11["median"],
                       "k11_distance_equals_solve_depth": bool(torch.equal(ds.cpu(), res.solve_depth_per_puzzle.cpu().int()))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    from tiler_slider_b200.generate import fill
    E = ts.BatchedTilerSliderEnv
    out = {"card": card(), "envs": args.envs, "reps": args.reps, "batches": {}}
    work = [("6x6_5_tiles_8_walls_coloured_solvable_8_12", 6, 5, 8, True),
            ("6x6_5_tiles_8_walls_coloured_synthetic", 6, 5, 8, False),
            ("8x8_5_tiles_12_walls_coloured_solvable_8_12", 8, 5, 12, True),
            ("6x6_6_tiles_8_walls_coloured_solvable_8_12", 6, 6, 8, True)]
    for key, S, T, W, graded in work:
        try:
            if graded:
                stats_of_fill = {}

                def gen():
                    env = E(S, T, args.envs, True)           # solvable()'s own steps, keeping fill's statistics
                    stats_of_fill.update(fill(env, W, min_depth=8, max_depth=12, recipe="walk", walk_len=24, seed=1,
                                              env_index_base=0, max_attempts=4096))
                    env._loaded = True
                    env.reset()
                    return env
                env, gen_s = timed(gen, args.reps)
                g = {"generate_s": gen_s, **stats_of_fill, "yield": stats_of_fill["accepted"] / stats_of_fill["candidates"],
                     "accepted_per_s_median": stats_of_fill["accepted"] / gen_s["median"]}
                assert stats_of_fill["unfilled"] == 0
            else:
                env, g = E.synthetic(args.envs, S, T, W, True, seed=1), None
            r = run_batch(env, args.reps, args.baseline)
            if g is not None:
                r = {"generate": g, **r}
        except Exception as e:                           # keep the other workloads' numbers
            r = {"error": repr(e)}
        out["batches"][key] = r
        print(key, json.dumps(r), flush=True)
        env = None
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
