"""Hash-table state tables (state_table(hash_table=True), K12 ts_state_table_count_table +
ts_state_table_fill_table) for 5 and 6 tiles, against labelling the same rows with the hash-table
optimal-move query (optimal_moves(ids, pos, hash_table=True), K11), which is what the labels cost once
the states are known.

  python profiles/experiments/table_state_table.py --out /tmp/table_state_table.json

Batches, at episode start:
  4,096 envs of 6x6 / 5 tiles / 8 walls, coloured, solvable() [8, 12]
  4,096 envs of 6x6 / 5 tiles / 8 walls, coloured, synthetic() (mostly unsolvable)
  4,096 envs of 6x6 / 5 tiles / 8 walls, single colour, solvable() [8, 12]
  256 envs of 6x6 / 6 tiles / 8 walls, coloured, solvable() [8, 12], with max_states the largest
      item's state count (found by a first call with a bound of 2^22), so that no item is -3
Per batch, after one warm-up, every repetition times:
  table   state_table(hash_table=True): CUDA events around the count and the fill launch, and a host
          clock around the whole call (which reads the row count back); rows x rounds swept by the
          fill pass (counters[2]) beside each fill time.
Then once, the baseline:
  k11     optimal_moves(ids, pos, hash_table=True) on the table's rows in chunks of CHUNK rows (host
          clock around the loop, which ends in a device synchronise), with K11's bound raised to the
          table's where it is larger; the rows of the first items up to --baseline-rows rows (the
          synthetic rows are mostly dead states, each of which K11 searches to exhaustion), as rows/s.
Checks: K11's labels of those rows equal the table's, and every table call returns the same table.
Reported: median / min / max per quantity.
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

CHUNK = 1 << 20
PASSES = ("ts_state_table_count_table", "ts_state_table_fill_table")


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


class EventLib:
    """The library with CUDA events recorded around the two K12 launches (on the current stream)."""

    def __init__(self, lib):
        self._lib, self.ms = lib, {}

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if name not in PASSES:
            return f
        import torch

        def timed(*args):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = f(*args)
            e1.record()
            self.ms[name] = (e0, e1)
            return rc
        return timed


def stats(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def k11_labeller(env, max_states):
    """K11 on env with a bound of at least max_states discovered states (grid within 4 GiB)."""
    from tiler_slider_b200.bfs import CudaOptimalMoves
    q = CudaOptimalMoves(env)
    if max_states is not None and max_states > q._plan_table()["spill_per_cta"]:
        q = CudaOptimalMoves(env, table_slots=1 << (2 * max_states - 1).bit_length())
        plan = q._plan_table()
        plan["grid"] = max(1, min(plan["grid"], q.MAX_SCRATCH_BYTES // (12 * plan["table_slots"])))
    return q


def run_batch(env, reps, max_states, baseline_rows):
    import torch
    from tiler_slider_b200.bfs import CudaStateTable
    k12 = CudaStateTable(env)
    k12.lib = ev = EventLib(k12.lib)
    env._state_table = k12

    def table():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tab = env.state_table(hash_table=True, max_states=max_states)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        count, fill = (ev.ms[p][0].elapsed_time(ev.ms[p][1]) / 1e3 for p in PASSES)
        return tab, wall, count, fill, int(k12.counters[2])

    tab, *_ = table()                                    # warm-up
    M = int(tab.offsets[-1])
    walls, counts, fills, swept, same = [], [], [], [], True
    for _ in range(reps):
        t2, w, c, f, s = table()
        same &= all(torch.equal(getattr(t2, k), getattr(tab, k)) for k in ("offsets", "status", "pos", "distance", "mask"))
        walls.append(w); counts.append(c); fills.append(f); swept.append(s)
    plan = k12._plan_table(max_states)

    # baseline: K11 on the rows of the first items, up to baseline_rows rows
    off = tab.offsets.cpu()
    n_items = max(1, int(torch.searchsorted(off, torch.tensor([baseline_rows]), right=True)) - 1)
    B = int(off[n_items]) if M else 0
    ids = torch.repeat_interleave(torch.arange(env.n_envs, device="cuda"), tab.offsets.diff())[:B].to(torch.int32)
    chunks = [(ids[i:i + CHUNK].contiguous(), tab.pos[i:i + CHUNK].contiguous()) for i in range(0, B, CHUNK)]
    k11 = k11_labeller(env, max_states)
    equal = True
    if chunks:
        k11.query(chunks[0][0][:4096], 254, chunks[0][1][:4096].contiguous(), hash_table=True)    # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k, (i, p) in enumerate(chunks):
        d, m = k11.query(i, 254, p, hash_table=True)
        equal &= bool(torch.equal(d, tab.distance[k * CHUNK:k * CHUNK + len(i)])
                      and torch.equal(m, tab.mask[k * CHUNK:k * CHUNK + len(i)]))
    torch.cuda.synchronize()
    t_k11 = time.perf_counter() - t0
    dist = tab.distance
    return {
        "envs": env.n_envs, "max_states": max_states, "rows": M, "rows_per_item_mean": M / env.n_envs,
        "status": {str(k): int((tab.status == k).sum()) for k in (0, -3, -4)},
        "rows_won_reachable": int((dist > 0).sum()), "max_distance": int(dist.max()) if M else None,
        "plan": {k: plan[k] for k in ("grid", "ctas_per_sm", "queue_smem", "table_slots", "spill_per_cta")},
        "count_pass_s": stats(counts), "fill_pass_s": stats(fills), "rows_x_rounds_swept": swept,
        "state_table_call_s": stats(walls), "table_rows_per_s_median": M / statistics.median(walls),
        "every_call_same_table": same,
        "baseline": {"items": n_items, "rows": B, "k11_chunk": CHUNK, "k11_s": t_k11,
                     "k11_rows_per_s": B / t_k11 if B else None,
                     "table_rows_per_s_over_k11_rows_per_s": (M / statistics.median(walls)) / (B / t_k11) if B else None,
                     "k11_labels_equal_table": equal},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--envs6", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-rows", type=int, default=4 << 20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    E = ts.BatchedTilerSliderEnv
    out = {"card": card(), "reps": args.reps, "batches": {}}
    work = [("6x6_5_tiles_8_walls_coloured_solvable_8_12", lambda: E.solvable(args.envs, 6, 5, 8, True, min_depth=8, max_depth=12, seed=1, hash_table=True), None),
            ("6x6_5_tiles_8_walls_coloured_synthetic", lambda: E.synthetic(args.envs, 6, 5, 8, True, seed=1), None),
            ("6x6_5_tiles_8_walls_single_colour_solvable_8_12", lambda: E.solvable(args.envs, 6, 5, 8, False, min_depth=8, max_depth=12, seed=1, hash_table=True), None),
            ("6x6_6_tiles_8_walls_coloured_solvable_8_12", lambda: E.solvable(args.envs6, 6, 6, 8, True, min_depth=8, max_depth=12, seed=1, hash_table=True), "fit")]
    for key, make, bound in work:
        try:
            env = make()
            if bound == "fit":                           # the smallest bound that leaves no item -3
                probe = env.state_table(hash_table=True, max_states=1 << 22)
                assert (probe.status == 0).all(), "an item reaches more than 2^22 states"
                bound = int(probe.offsets.diff().max())
                probe = None
            r = run_batch(env, args.reps, bound, args.baseline_rows)
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
