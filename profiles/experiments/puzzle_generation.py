"""Puzzle generation and pool-reset measurements (BatchedTilerSliderEnv.solvable, set_reset_pool).

  python profiles/experiments/puzzle_generation.py --out /tmp/puzzle_generation.json
      (a) generation rate on one GPU: accepted puzzles/s and candidates/s for 6x6 / 4 tiles / 8 walls,
          coloured and single-colour, recipes walk and uniform, bands [1,30], [8,12], [12,20]
          (65,536 envs; host clock around rounds that end in a device synchronise; the uniform
          recipe is stopped after --uniform-rounds rounds, the walk fills every env);
      (b) the c3 step (6x6 / 4 coloured tiles / 8 walls, 16.7M envs, auto-reset, no status byte) with
          and without an attached 65,536-puzzle pool, bench.py's method: 50-step CUDA graphs, CUDA
          events, a clock ramp first, the two batches alternated block by block.
  python profiles/experiments/puzzle_generation.py --cpu-walk-yield --out walk_yield.json
      share of walk candidates (C oracle BFS) in each band for several walk lengths, on the CPU.
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

BANDS = [(1, 30), (8, 12), (12, 20)]


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def generation(args):
    import torch
    import tiler_slider_b200 as ts
    from tiler_slider_b200.generate import default_walk_len, fill
    S, T, W, N = 6, 4, 8, args.gen_envs
    rows = []
    for multi in (True, False):
        warm = ts.BatchedTilerSliderEnv(S, T, 4096, multi)
        fill(warm, W, min_depth=1, max_depth=30, recipe="walk", walk_len=60, seed=1, env_index_base=0, max_attempts=2)
        for recipe in ("walk", "uniform"):
            for lo, hi in BANDS:
                env = ts.BatchedTilerSliderEnv(S, T, N, multi)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = fill(env, W, min_depth=lo, max_depth=hi, recipe=recipe, walk_len=default_walk_len(hi), seed=2024,
                          env_index_base=0, max_attempts=args.uniform_rounds if recipe == "uniform" else 4096)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                rows.append(dict(multi=multi, recipe=recipe, band=[lo, hi], walk_len=default_walk_len(hi) if recipe == "walk" else None,
                                 envs=N, seconds=dt, **st, accepted_per_s=st["accepted"] / dt,
                                 candidates_per_s=st["candidates"] / dt, yield_fraction=st["accepted"] / st["candidates"]))
                print(json.dumps(rows[-1]), flush=True)
    return rows


def pool_step(args):
    import torch
    import tiler_slider_b200 as ts
    N, K, R = args.step_envs, 50, 8
    pool = ts.BatchedTilerSliderEnv.solvable(65536, 6, 4, 8, True, min_depth=1, max_depth=30, seed=7)
    kw = dict(seed=1002, max_steps=100, auto_reset=True, track_flags=False)
    plain = ts.BatchedTilerSliderEnv.synthetic(N, 6, 4, 8, True, **kw)
    pooled = ts.BatchedTilerSliderEnv.synthetic(N, 6, 4, 8, True, **kw)
    pooled.set_reset_pool(pool, seed=3, draw_now=True)
    gen = torch.Generator(device="cuda").manual_seed(2002)
    actions = torch.randint(0, 4, (R, plain.capacity), dtype=torch.uint8, device="cuda", generator=gen)
    rows = actions[torch.arange(K, device="cuda") % R].contiguous()
    graphs = {"plain": plain.capture_steps(rows), "pool": pooled.capture_steps(rows)}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    busy = 0.0
    while busy < 300.0:                                        # clock ramp
        ev[0].record()
        for g in graphs.values():
            g.replay()
        ev[1].record()
        ev[1].synchronize()
        busy += ev[0].elapsed_time(ev[1])
    ep0 = int(pooled.episodes.to(torch.int64).sum())
    times = {"plain": [], "pool": []}
    for rep in range(args.blocks):
        for name in (("plain", "pool") if rep % 2 == 0 else ("pool", "plain")):
            ev[0].record()
            for _ in range(args.graphs_per_block):
                graphs[name].replay()
            ev[1].record()
            ev[1].synchronize()
            times[name].append(ev[0].elapsed_time(ev[1]) / (K * args.graphs_per_block))
    draws = int(pooled.episodes.to(torch.int64).sum()) - ep0
    steps = args.blocks * args.graphs_per_block * K
    out = {k: dict(ms_per_step_median=statistics.median(v), ms_per_step_min=min(v), ms_per_step_max=max(v), blocks=v)
           for k, v in times.items()}
    out.update(envs=N, pool_puzzles=65536, steps_per_block=K * args.graphs_per_block,
               pool_draws_per_env_step=draws / (steps * N),
               extra_us_per_step_median=1e3 * (out["pool"]["ms_per_step_median"] - out["plain"]["ms_per_step_median"]))
    print(json.dumps({k: v for k, v in out.items() if k not in ("plain", "pool")}), flush=True)
    return out


def cpu_walk_yield(args):
    import numpy as np
    from oracle import oracle as orc
    from tests import gen_port
    S, T, W = 6, 4, 8
    out = []
    for multi in (True, False):
        for walk_len in (8, 20, 40, 60):
            depths = []
            for g in range(args.cpu_puzzles):
                b, tiles, targets = gen_port.candidate(orc, S, T, W, multi, "walk", walk_len, 2024, 0, g)
                st = orc.OracleState(S, [divmod(c, S) for c in b], tiles, targets, multi)
                depths.append(st.bfs(max_depth=64, max_states=1 << 20)[2])
            d = np.array(depths)
            row = dict(multi=multi, walk_len=walk_len, puzzles=len(d), median=float(np.median(d)),
                       p90=float(np.percentile(d, 90)),
                       in_band={f"{lo}-{hi}": float(((d >= lo) & (d <= hi)).mean()) for lo, hi in BANDS})
            out.append(row)
            print(json.dumps(row), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gen-envs", type=int, default=65536)
    ap.add_argument("--uniform-rounds", type=int, default=200)
    ap.add_argument("--step-envs", type=int, default=16_777_216)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--graphs-per-block", type=int, default=4)
    ap.add_argument("--cpu-walk-yield", action="store_true")
    ap.add_argument("--cpu-puzzles", type=int, default=200)
    args = ap.parse_args()
    if args.cpu_walk_yield:
        res = {"what": "walk recipe, 6x6 / 4 tiles / 8 walls: C oracle BFS solve depth of walk candidates (CPU)",
               "rows": cpu_walk_yield(args)}
    else:
        import torch
        if not torch.cuda.is_available():
            raise SystemExit("needs a GPU")
        res = {"card": card(), "generation": generation(args), "pool_step": pool_step(args)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
