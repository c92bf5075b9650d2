"""State tables (env.state_table(), K10 ts_state_table_count + ts_state_table_fill) against labelling
the same rows with the optimal-move query (optimal_moves(ids, pos), K9), which is what the labels
cost once the states are known.

  python profiles/experiments/state_table.py --out /tmp/state_table.json

65,536 envs of 6x6 / 4 tiles / 8 walls at episode start: coloured solvable() [8, 12], coloured
synthetic() (mostly unsolvable: the fill pass skips the sweep) and single-colour solvable() [8, 12].
Per batch, after one warm-up of each, every repetition times in turn:
  table   state_table(): CUDA events around the count and the fill launch, and a host clock around
          the whole call (which reads the free-cell maximum and the row count back);
  k9      optimal_moves(ids, pos) on every row of that table, in chunks of CHUNK rows (host clock
          around the whole loop, which ends in a device synchronise), as rows/s.
Checks: the K9 labels of every row equal the table's, and every table call returns the same table.
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

CHUNK = 1 << 22


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


class EventLib:
    """The library with CUDA events recorded around the two K10 launches (on the current stream)."""

    def __init__(self, lib):
        self._lib, self.ms = lib, {}

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if name not in ("ts_state_table_count", "ts_state_table_fill"):
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


def run_batch(env, reps):
    import torch
    from tiler_slider_b200.bfs import CudaStateTable
    k10 = CudaStateTable(env)
    k10.lib = ev = EventLib(k10.lib)
    env._state_table = k10

    def table():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tab = env.state_table()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        count = ev.ms["ts_state_table_count"][0].elapsed_time(ev.ms["ts_state_table_count"][1]) / 1e3
        fill = ev.ms["ts_state_table_fill"][0].elapsed_time(ev.ms["ts_state_table_fill"][1]) / 1e3
        return tab, wall, count, fill

    tab, *_ = table()                                    # warm-up
    M = int(tab.offsets[-1])
    ids = torch.repeat_interleave(torch.arange(env.n_envs, device="cuda"), tab.offsets.diff()).to(torch.int32)
    chunks = [(ids[i:i + CHUNK].contiguous(), tab.pos[i:i + CHUNK].contiguous()) for i in range(0, M, CHUNK)]

    def k9(check=False):
        """Every row labelled by K9, chunk by chunk; check: compare each chunk with the table."""
        equal = True
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k, (i, p) in enumerate(chunks):
            d, m = env.optimal_moves(i, pos=p)
            if check:
                equal &= bool(torch.equal(d, tab.distance[k * CHUNK:k * CHUNK + len(i)])
                              and torch.equal(m, tab.mask[k * CHUNK:k * CHUNK + len(i)]))
        torch.cuda.synchronize()
        return time.perf_counter() - t0, equal

    _, labels_equal = k9(check=True)                     # warm-up, and the check
    walls, counts, fills, k9s = [], [], [], []
    for _ in range(reps):
        t2, w, c, f = table()
        assert torch.equal(t2.pos, tab.pos) and torch.equal(t2.distance, tab.distance)
        walls.append(w); counts.append(c); fills.append(f)
        k9s.append(k9()[0])
    dist = tab.distance
    return {
        "envs": env.n_envs, "rows": M, "rows_per_item_mean": M / env.n_envs,
        "status_nonzero": int((tab.status != 0).sum()),
        "rows_won_reachable": int((dist > 0).sum()), "max_distance": int(dist.max()) if M else None,
        "rows_swept": int(k10.counters[2]),
        "count_pass_s": stats(counts), "fill_pass_s": stats(fills), "state_table_call_s": stats(walls),
        "table_rows_per_s_median": M / statistics.median(walls),
        "k9_all_rows_s": stats(k9s), "k9_rows_per_s_median": M / statistics.median(k9s),
        "k10_speedup_median": statistics.median(k9s) / statistics.median(walls),
        "k9_labels_equal_table_every_row": labels_equal,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import tiler_slider_b200 as ts
    E = ts.BatchedTilerSliderEnv
    out = {"card": card(), "shape": "6x6, 4 tiles, 8 walls", "k9_chunk": CHUNK, "batches": {}}
    for name, make in (("coloured_solvable_8_12", lambda: E.solvable(args.envs, 6, 4, 8, True, min_depth=8, max_depth=12, seed=1)),
                       ("coloured_synthetic", lambda: E.synthetic(args.envs, 6, 4, 8, True, seed=1)),
                       ("single_colour_solvable_8_12", lambda: E.solvable(args.envs, 6, 4, 8, False, min_depth=8, max_depth=12, seed=1))):
        out["batches"][name] = r = run_batch(make(), args.reps)
        print(name, json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
