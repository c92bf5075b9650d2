"""Does alternating the step's env traversal order let each step reuse what the previous one left in
L2?  Ascending-only against alternating ts_step_args.order, in one process and one build.

  python profiles/experiments/l2_reuse.py --out profiles/r8_l2_reuse_b200.json

Per row (bench.py's c3 / c4 puzzles, max_steps 100, auto-reset on, 1-byte counters, no flags -- the
launch bench.py times), on the same batch:
  ascending    every launch walks the envs from first to last (order 0, the behaviour before the field)
  alternating  launch k walks them in order k % 2, as BatchedTilerSliderEnv.step() does
Each variant is a CUDA graph of --block ts_step launches (action row k % 8 for launch k, as bench.py);
a round times one replay of each variant with CUDA events, in alternating order, after a clock ramp of
--ramp-ms busy time per row; the median over --rounds rounds is reported, with its spread.
Mechanism check: alternation can only gain where the bytes one step touches are larger than the L2
(126 MB) and the L2 can still hold a useful share of them, so the gain should be nil while the
working set fits the L2 (2 M c3 envs, about 55 MB per step), largest at a small multiple of it, and
shrink again as the share the L2 holds falls (33.5 M c3 envs).  bytes_per_step is what one launch
requests (BYTES_PER_ENV below); working_set_over_l2 sets it against the 126 MB L2.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

# name, size, tiles, walls, multi, puzzle seed, action seed (bench.py's CONFIGS)
CONFIGS = {"c3": (6, 4, 8, True, 1002, 2002), "c4": (12, 8, 36, True, 1003, 2003)}
SWEEP = [("c3", n) for n in (2_097_152, 4_194_304, 6_291_456, 8_388_608, 16_777_216, 33_554_432)] + \
        [("c4", n) for n in (1_048_576, 2_097_152, 4_194_304, 8_388_608)]
# bytes one launch requests per env, reads + writes (DESIGN.md sections 3 and 4): c3 16 B read + 10 B
# written; c4 64 B read + 19 B written
BYTES_PER_ENV = {"c3": 26, "c4": 83}
N_ACTION_ROWS = 8
VARIANTS = ("ascending", "alternating")


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def capture(lib, args, rows, orders, stream_of):
    """One CUDA graph of len(orders) ts_step launches; launch k uses action row k % len(rows)."""
    import torch
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        s = stream_of()
        for k, o in enumerate(orders):
            args.d_actions = rows[k % len(rows)].data_ptr()
            args.order = o
            rc = lib.ts_step(C.byref(args), s)
            if rc:
                raise RuntimeError(f"ts_step: {rc}")
    return g


def row(ts, lib, name, n, block, rounds, ramp_ms):
    import torch
    S, T, W, multi, pseed, aseed = CONFIGS[name]
    env = ts.BatchedTilerSliderEnv.synthetic(n, S, T, W, multi, seed=pseed, max_steps=100, auto_reset=True,
                                             track_flags=False, device="cuda:0")
    gen = torch.Generator(device="cuda:0").manual_seed(aseed)
    rows = torch.randint(0, 4, (N_ACTION_ROWS, env.capacity), dtype=torch.uint8, device="cuda:0", generator=gen)
    args = env._step_args(rows[0].data_ptr())
    stream_of = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    graphs = {"ascending": capture(lib, args, rows, [0] * block, stream_of),
              "alternating": capture(lib, args, rows, [k % 2 for k in range(block)], stream_of)}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    busy = 0.0
    while busy < ramp_ms:                       # clock ramp; also uploads both graphs
        for g in graphs.values():
            ev[0].record(); g.replay(); ev[1].record(); ev[1].synchronize()
            busy += ev[0].elapsed_time(ev[1])
    times = {v: [] for v in VARIANTS}
    for r in range(rounds):
        for v in (VARIANTS if r % 2 == 0 else VARIANTS[::-1]):
            ev[0].record(); graphs[v].replay(); ev[1].record(); ev[1].synchronize()
            times[v].append(ev[0].elapsed_time(ev[1]) * 1e3 / block)
    out = {"config": name, "envs": n, "bytes_per_step": BYTES_PER_ENV[name] * n,
           "working_set_over_l2": round(BYTES_PER_ENV[name] * n / 126e6, 2)}
    for v in VARIANTS:
        t = sorted(times[v])
        out[v] = {"us_per_step_median": round(statistics.median(t), 3), "us_min": round(t[0], 3), "us_max": round(t[-1], 3),
                  "dram_equiv_TBps": round(BYTES_PER_ENV[name] * n / statistics.median(t) / 1e6, 3)}
    out["gain_alternating_pct"] = round(100 * (out["ascending"]["us_per_step_median"] / out["alternating"]["us_per_step_median"] - 1), 2)
    del graphs, env, rows
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_l2_reuse_b200.json"))
    ap.add_argument("--block", type=int, default=200, help="launches per timed graph (even: the alternating graph ends where it started)")
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--ramp-ms", type=float, default=150.0)
    ap.add_argument("--only", help="comma-separated config:envs rows, e.g. c3:16777216")
    a = ap.parse_args()
    if a.block < 200 or a.block % 2:
        ap.error("--block must be an even number >= 200")
    import torch
    if not torch.cuda.is_available():
        sys.exit("l2_reuse.py measures on the GPU; no CUDA device found")
    import tiler_slider_b200 as ts
    from tiler_slider_b200 import _lib
    torch.cuda.set_device(0)
    lib = _lib.lib()
    sweep = SWEEP if not a.only else [(c.split(":")[0], int(c.split(":")[1])) for c in a.only.split(",")]
    res = {"what": "ts_step, ascending-only vs alternating traversal order (ts_step_args.order)",
           "how": f"CUDA graphs of {a.block} launches per variant, {a.rounds} rounds alternating the variants, "
                  f"median us per launch; {a.ramp_ms:.0f} ms clock ramp per row",
           "card_before": card(), "rows": []}
    for name, n in sweep:
        r = row(ts, lib, name, n, a.block, a.rounds, a.ramp_ms)
        print(json.dumps(r), flush=True)
        res["rows"].append(r)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
