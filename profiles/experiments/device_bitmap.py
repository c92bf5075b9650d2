"""Device-memory bitmaps (device_bitmap=True): 7x7 and 8x8 boards with four tiles whose state space
outgrows one CTA's shared memory, searched by K6 (solvable(), LocalBfs), K9 (optimal_moves) and K10
(state_table) with the bitmap in device memory.

  python profiles/experiments/device_bitmap.py --out /tmp/device_bitmap.json

Workloads: 65,536 envs of 7x7 / 4 tiles / 8 walls and of 8x8 / 4 tiles / 12 walls, coloured, at
episode start: solvable() [8, 12] and synthetic().  Every timing is a host clock around a call that
ends in a device synchronise; after one warm-up, `--reps` repetitions, reported as median / min / max.
  generate     solvable(..., device_bitmap=True) (the solvable() batch only; K7 + K6 rounds)
  k9           optimal_moves(device_bitmap=True), without and with paths
  k10          state_table(device_bitmap=True): CUDA events around the count and the fill launch,
               and rows/s of the whole call
  k6           LocalBfs(device_bitmap=True).solve(), as successors generated per second
Beside each time: the bytes the whole-bitmap clears write per item (F!/(F-4)!/8 per clear: K9 two
when distance >= 2, K6 one, K10 one in count and two in fill when a win is reachable, plus one read
by the fill's order scan), summed over the batch, since those may dominate the time.

The cost of the device bitmap: 7x7 / 4 tiles / 12 walls (F = 37, which fits both instances), K9 and
K10 on the shared plan and on the forced gmem plan, alternated in one run; the answers are compared.
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


def clear_bytes(env):
    """Bytes one whole-bitmap clear writes, per env (F!/(F-T)! bits rounded up to 16-byte units)."""
    F = (env.size * env.size - env.blocked_cells().sum(1)).long()
    bits = F * (F - 1) * (F - 2) * (F - 3)
    return ((bits + 127) // 128) * 16


class EventLib:
    """The library with CUDA events recorded around the two K10 launches (on the current stream)."""

    def __init__(self, lib):
        self._lib, self.ms = lib, {}

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if not name.startswith("ts_state_table_count") and not name.startswith("ts_state_table_fill"):
            return f
        import torch

        def run(*args):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = f(*args)
            e1.record()
            self.ms["fill" if "fill" in name else "count"] = (e0, e1)
            return rc
        return run


def run_batch(env, reps):
    import torch
    from tiler_slider_b200.bfs import CudaStateTable, LocalBfs
    n = env.n_envs
    cb = clear_bytes(env)
    out = {"envs": n, "free_cells_min_max": [int(x) for x in torch.aminmax(env.size * env.size - env.blocked_cells().sum(1))],
           "clear_bytes_per_item_mean": float(cb.double().mean())}
    (d, m), out["k9_s"] = timed(lambda: env.optimal_moves(device_bitmap=True), reps)
    out["k9_status_not_searched"] = int((d == -3).sum())
    out["k9_solved"] = int((d >= 1).sum())
    out["k9_clear_bytes"] = int((cb * (1 + (d >= 2).long())).sum())
    (dp, mp, _), out["k9_paths_s"] = timed(lambda: env.optimal_moves(paths=True, device_bitmap=True), reps)
    out["k9_paths_equal_no_paths"] = bool(torch.equal(d, dp) and torch.equal(m, mp))

    k10 = CudaStateTable(env)
    k10.lib = ev = EventLib(k10.lib)
    env._state_table = k10
    counts, fills = [], []

    def table():
        tab = env.state_table(device_bitmap=True)
        torch.cuda.synchronize()
        counts.append(ev.ms["count"][0].elapsed_time(ev.ms["count"][1]) / 1e3)
        fills.append(ev.ms["fill"][0].elapsed_time(ev.ms["fill"][1]) / 1e3)
        return tab
    tab, out["k10_call_s"] = timed(table, reps)
    counts, fills = counts[1:], fills[1:]
    M = int(tab.offsets[-1])
    swept = (tab.distance >= 1).any()
    out.update(k10_rows=M, k10_rows_per_item_mean=M / n, k10_status_nonzero=int((tab.status != 0).sum()),
               k10_count_pass_s=stats(counts), k10_fill_pass_s=stats(fills),
               k10_rows_per_s_median=M / out["k10_call_s"]["median"],
               k10_clear_bytes_count=int(cb.sum()),
               k10_clear_and_scan_bytes_fill=int(cb.sum()) * (3 if bool(swept) else 2))

    res, out["k6_s"] = timed(lambda: LocalBfs(env, device_bitmap=True).solve(per_puzzle=False), reps)
    out.update(k6_fallback_puzzles=res.fallback_puzzles, k6_states=res.n_states, k6_successors=res.generated,
               k6_successors_per_s_median=res.generated / out["k6_s"]["median"], k6_clear_bytes=int(cb.sum()))
    return out


def cost_of_device_bitmap(E, n, reps):
    """7x7 / 4 / 12 walls: K9 and K10 on the shared plan and on the forced gmem plan, alternated."""
    import torch
    from tiler_slider_b200.bfs import CudaOptimalMoves, CudaStateTable

    def forced(cls):
        class Forced(cls):
            def plan(self, f_max):
                p = super().plan(f_max)
                return None if p is None else self._plan_gmem(p["f_max"])
        return Forced

    env = E.solvable(n, 7, 4, 12, True, min_depth=8, max_depth=12, seed=3)
    runs = {"k9_shared": CudaOptimalMoves(env).query, "k9_gmem": forced(CudaOptimalMoves)(env).query}
    k10s, k10g = CudaStateTable(env), forced(CudaStateTable)(env)
    plans = {"k9_shared": CudaOptimalMoves(env).plan(37), "k9_gmem": forced(CudaOptimalMoves)(env).plan(37)}
    res = {k: [] for k in ("k9_shared", "k9_gmem", "k10_shared", "k10_gmem")}
    last = {}
    calls = {"k9_shared": lambda: runs["k9_shared"](None, 254), "k9_gmem": lambda: runs["k9_gmem"](None, 254),
             "k10_shared": lambda: k10s.build(None), "k10_gmem": lambda: k10g.build(None)}
    for k, f in calls.items():                            # warm-up
        last[k] = f()
    for _ in range(reps):
        for k, f in calls.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            last[k] = f()
            torch.cuda.synchronize()
            res[k].append(time.perf_counter() - t0)
    return {"shape": "7x7, 4 tiles, 12 walls (F = 37), coloured solvable() [8, 12]", "envs": n,
            "plans": {k: {x: v for x, v in p.items() if x != "smem_bytes"} for k, p in plans.items()},
            "times_s": {k: stats(v) for k, v in res.items()},
            "gmem_over_shared_median": {"k9": statistics.median(res["k9_gmem"]) / statistics.median(res["k9_shared"]),
                                        "k10": statistics.median(res["k10_gmem"]) / statistics.median(res["k10_shared"])},
            "k9_answers_equal": all(torch.equal(a, b) for a, b in zip(last["k9_shared"], last["k9_gmem"])),
            "k10_tables_equal": all(torch.equal(a, b) for a, b in zip(last["k10_shared"], last["k10_gmem"])),
            "clear_bytes_per_item": int(clear_bytes(env)[0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    E = ts.BatchedTilerSliderEnv
    out = {"card": card(), "envs": args.envs, "reps": args.reps, "batches": {}}
    for S, W in ((7, 8), (8, 12)):
        gen = lambda: E.solvable(args.envs, S, 4, W, True, min_depth=8, max_depth=12, seed=1, device_bitmap=True)
        env, gen_s = timed(gen, args.reps)
        batches = {"coloured_solvable_8_12": (env, gen_s), "coloured_synthetic": (E.synthetic(args.envs, S, 4, W, True, seed=1), None)}
        for name, (b, g) in batches.items():
            key = f"{S}x{S}_4_tiles_{W}_walls_{name}"
            r = run_batch(b, args.reps)
            if g is not None:
                r = {"generate_s": g, **r}
            out["batches"][key] = r
            print(key, json.dumps(r), flush=True)
            del b
        del env, batches
        torch.cuda.empty_cache()
    out["cost_of_device_bitmap"] = c = cost_of_device_bitmap(E, args.envs, args.reps + 2)
    print("cost_of_device_bitmap", json.dumps(c), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
