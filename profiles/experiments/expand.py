"""Throughput of ts_expand (BatchedTilerSliderEnv.expand) beside what a user pays today for the same
successors, and of observe_planes() of the 4N successors beside observe_planes() of the N envs.

  python profiles/experiments/expand.py --out /tmp/expand.json

Shapes (synthetic() puzzles; every timed output larger than the 126 MB L2):
  6x6 / 4 tiles / 8 walls multi-colour at 16,777,216 items, dense (ids None) and with shuffled ids
  (a random permutation, int32 on the device); 5x5 / 1 tile / 5 walls single-colour at 33,554,432
  items; 8x8 / 4 tiles / 12 walls multi-colour at 16,777,216; 12x12 / 8 tiles / 36 walls
  multi-colour at 4,194,304 (wide kernel); 8x8 / 12 tiles / 10 walls multi-colour at 4,194,304
  (generic kernel).
Per row, on the same batch in the same run:
  expand    expand(ids, out=...) into preallocated outputs;
  composed  today's composition: clone pos; four times (restore pos, raw_move(a) with a
            preallocated action row, copy pos and the flags out); restore pos.  Its successors,
            moved (!INVALID) and won (WON) bits are checked equal to expand()'s before timing.
Algorithmic bytes per item (computed below from the shape): ids (4, when listed) + the position
word + the env's walls (bitboard bytes; wide boards: both axis records) + its targets (ordered: a
position word; set: the target board) read, 4 successor words + the two mask bytes written.
Planes: observe_planes(bf16) of the 4N successors (ids.repeat_interleave(4), succ.reshape(-1, PW))
against observe_planes(bf16) of the N envs, 6x6 / 4 tiles at N = 1,048,576 and 12x12 / 8 tiles at
N = 262,144.
Timing: CUDA events around `--calls` back-to-back calls after 3 warm-up calls, `--rounds` rounds
alternating the variants; the median round is reported.  Card name, power limit and clocks are read
in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

# (S, T, walls, multi, items, shuffled ids)
SHAPES = [(6, 4, 8, True, 16_777_216, False), (6, 4, 8, True, 16_777_216, True), (5, 1, 5, False, 33_554_432, False),
          (8, 4, 12, True, 16_777_216, False), (12, 8, 36, True, 4_194_304, False), (8, 12, 10, True, 4_194_304, False)]
PLANE_SHAPES = [(6, 4, 8, True, 1_048_576), (12, 8, 36, True, 262_144)]
F_WON, F_INVALID = 2, 4


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def time_calls(fn, calls):
    import torch
    for _ in range(3):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(calls):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / calls


def item_bytes(env, listed):
    """Algorithmic bytes per item: what the kernel must read and write."""
    lib = env._lib
    PW = env.pos_bytes
    walls = lib.ts_walls_bytes(env.size)                 # wide boards: both axis records (the four moves use both)
    targets = PW if env.goal_mode == 0 else lib.ts_target_board_bytes(env.size)
    return (4 if listed else 0) + PW + walls + targets + 4 * PW + 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=int, default=1, help="divide the item counts (rehearsal only)")
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    if not torch.cuda.is_available():
        raise SystemExit("expand.py measures on a GPU; none found")
    res = {"card": card(), "calls": args.calls, "rounds": args.rounds, "rows": [], "planes": []}
    for S, T, W, multi, N, shuffled in SHAPES:
        N //= args.scale
        env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=1)
        g = torch.Generator(device="cuda").manual_seed(2)
        for _ in range(3):      # positions other than the initial ones
            env.raw_move(torch.randint(0, 4, (env.capacity,), dtype=torch.uint8, device="cuda", generator=g))
        PW = env.pos_bytes
        ids = torch.randperm(N, device="cuda", generator=g).to(torch.int32) if shuffled else None
        out = (torch.empty(N, 4, PW, dtype=torch.uint8, device="cuda"), torch.empty(N, dtype=torch.uint8, device="cuda"),
               torch.empty(N, dtype=torch.uint8, device="cuda"))
        saved = torch.empty_like(env._pos)
        c_succ = torch.empty(4, N, PW, dtype=torch.uint8, device="cuda")
        c_flags = torch.empty(4, N, dtype=torch.uint8, device="cuda")
        acts = [torch.full((env.capacity,), a, dtype=torch.uint8, device="cuda") for a in range(4)]

        def composed():
            saved.copy_(env._pos)
            for a in range(4):
                if a:
                    env._pos.copy_(saved)
                c_flags[a].copy_(env.raw_move(acts[a]))
                c_succ[a].copy_(env.pos)
            env._pos.copy_(saved)

        def expand():
            env.expand(ids, out=out)

        expand()
        composed()
        perm = ids.long() if shuffled else slice(None)
        bits = torch.arange(4, device="cuda", dtype=torch.uint8)[:, None]
        assert torch.equal(out[0], c_succ.transpose(0, 1)[perm]), (S, T)
        assert torch.equal(out[1], (((c_flags & F_INVALID) == 0).to(torch.uint8) << bits).sum(0, dtype=torch.uint8)[perm]), (S, T)
        assert torch.equal(out[2], (((c_flags & F_WON) != 0).to(torch.uint8) << bits).sum(0, dtype=torch.uint8)[perm]), (S, T)
        fns = {"expand": expand, "composed": composed}
        ms = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                ms[k].append(time_calls(fn, args.calls))
        med = {k: statistics.median(v) for k, v in ms.items()}
        b = item_bytes(env, shuffled)
        row = {"shape": f"{S}x{S}/{T} tiles/{W} walls {'multi' if multi else 'single'}-colour", "items": N,
               "ids": "shuffled" if shuffled else "none (dense)", "kernel": "generic" if T > 8 else ("wide" if S > 8 else "bitboard"),
               "algorithmic_bytes_per_item": b, "expand_ms": round(med["expand"], 4),
               "expand_items_per_s": N / med["expand"] * 1e3, "expand_gb_per_s": round(N * b / med["expand"] / 1e6, 1),
               "composed_ms": round(med["composed"], 4), "speedup_vs_composed": round(med["composed"] / med["expand"], 2),
               "rounds_ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}}
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
        del env, out, saved, c_succ, c_flags, acts, ids
        torch.cuda.empty_cache()
    for S, T, W, multi, N in PLANE_SHAPES:
        N //= args.scale
        env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=3)
        ids = torch.arange(N, dtype=torch.int32, device="cuda")
        succ, _, _ = env.expand(ids)
        ids4, pos4 = ids.repeat_interleave(4), succ.reshape(-1, env.pos_bytes)
        C = env.plane_count
        o_items = torch.empty(4 * N, C, S, S, dtype=torch.bfloat16, device="cuda")
        o_envs = torch.empty(N, C, S, S, dtype=torch.bfloat16, device="cuda")
        fns = {"items_4n": lambda: env.observe_planes(o_items, dtype=torch.bfloat16, ids=ids4, pos=pos4),
               "envs_n": lambda: env.observe_planes(o_envs, dtype=torch.bfloat16)}
        ms = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                ms[k].append(time_calls(fn, args.calls))
        med = {k: statistics.median(v) for k, v in ms.items()}
        img = C * S * S * 2
        row = {"shape": f"{S}x{S}/{T} tiles/{W} walls {'multi' if multi else 'single'}-colour", "envs": N, "dtype": "bfloat16",
               "bytes_per_image": img, "items_4n_ms": round(med["items_4n"], 4), "envs_n_ms": round(med["envs_n"], 4),
               "items_gb_written_per_s": round(4 * N * img / med["items_4n"] / 1e6, 1),
               "envs_gb_written_per_s": round(N * img / med["envs_n"] / 1e6, 1),
               "items_time_over_4x_envs_time": round(med["items_4n"] / (4 * med["envs_n"]), 3),
               "rounds_ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}}
        res["planes"].append(row)
        print(json.dumps(row), flush=True)
        del env, o_items, o_envs, succ
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
