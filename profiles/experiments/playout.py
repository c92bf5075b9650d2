"""Throughput of ts_playout (BatchedTilerSliderEnv.playout) beside what a user runs today for the same
playouts.

  python profiles/experiments/playout.py --out /tmp/playout.json

Rows (synthetic() puzzles, L = 64 moves, positions after 3 random moves; every timed working set but
the small-batch row is larger than the 126 MB L2):
  6x6 / 4 tiles / 8 walls multi-colour, 16,777,216 items: plan, plan with record=True, random;
  6x6 / 4 tiles, 65,536 items, random -- an MCTS-sized batch (small batch: its working set fits L2);
  5x5 / 1 tile / 5 walls single-colour, 33,554,432 items: plan, random;
  12x12 / 8 tiles / 36 walls multi-colour, 4,194,304 items (wide kernel): plan, random;
  8x8 / 12 tiles / 10 walls multi-colour, 4,194,304 items (generic kernel): plan, random.
Per row, on the same batch in the same run:
  fused     playout(out=...) into preallocated outputs (plan_record: with the moves and positions of every move);
  composed  today's composition: clone pos; per move raw_move(row k) (plan: the plan row; random:
            valid_moves(), a torch.rand draw among the set bits), then torch ops that freeze an item
            after its first WON (or the end of its plan / a state where nothing moves) and keep its
            positions and move count (plan_record: and stores the move and the positions of every move);
            restore pos.  Before timing it is checked to give the fused
            kernel's final / steps / won: for the plan on the same plan, for random on the moves the
            fused kernel recorded (each checked to be a valid move).
Reported: played moves/s (sum of steps over time), items/s, the time ratio, the algorithmic bytes per
item (computed below from the shape) and `-Xptxas -v` registers / spills of the kernels the rows run
(compiled from the sources in a temporary directory while the GPU measures).
Timing: CUDA events around `--calls` back-to-back calls after 2 warm-up calls, `--rounds` rounds
alternating the variants; the median round is reported.  Card name, power limit and clocks are read in
the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
CSRC = os.path.join(ROOT, "tiler_slider_b200", "csrc")

L = 64
# (S, T, walls, multi, items, policies, note)
ROWS = [(6, 4, 8, True, 16_777_216, ("plan", "plan_record", "random"), ""),
        (6, 4, 8, True, 65_536, ("random",), "small batch (MCTS-sized): working set fits L2"),
        (5, 1, 5, False, 33_554_432, ("plan", "random"), ""),
        (12, 8, 36, True, 4_194_304, ("plan", "random"), ""),
        (8, 12, 10, True, 4_194_304, ("plan", "random"), "")]
F_WON = 2


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def start_ptxas(tmp):
    """nvcc -Xptxas -v of the playout sources, in the background (the flags of csrc/Makefile)."""
    procs = {}
    for src in ("ts_playout.cu", "ts_wide.cu", "ts_generic.cu"):
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
               "-c", os.path.join(CSRC, src), "-o", os.path.join(tmp, src + ".o")]
        try:
            procs[src] = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        except OSError as e:
            procs[src] = str(e)
    return procs


def ptxas_report(procs):
    """{kernel (demangled template): registers / stack / spills} for the playout kernels."""
    out = {}
    for src, p in procs.items():
        if isinstance(p, str):
            out[src] = f"not measured: {p}"
            continue
        text = p.communicate()[0]
        cur = None
        for line in text.splitlines():
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                cur = m.group(1) if "playout" in m.group(1) else None
                continue
            if cur is None:
                continue
            m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
            if m:
                out.setdefault(cur, {}).update(stack=int(m.group(1)), spill_stores=int(m.group(2)), spill_loads=int(m.group(3)))
            m = re.search(r"Used (\d+) registers", line)
            if m:
                out.setdefault(cur, {})["registers"] = int(m.group(1))
    demangled = {}
    names = [k for k in out if isinstance(out[k], dict)]
    if names and shutil.which("cu++filt"):
        d = subprocess.run(["cu++filt"] + names, capture_output=True, text=True).stdout.splitlines()
        demangled = dict(zip(names, d))
    return {demangled.get(k, k): v for k, v in out.items()}


def time_calls(fn, calls):
    import torch
    for _ in range(2):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(calls):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / calls


def item_bytes(env, policy):
    """Algorithmic bytes per item: start positions, walls (wide boards: both axis records), targets and
    (plan) the L plan bytes read; final positions, steps and won written (record: L moves and L words)."""
    lib = env._lib
    PW = env.pos_bytes
    targets = PW if env.goal_mode == 0 else lib.ts_target_board_bytes(env.size)
    b = PW + lib.ts_walls_bytes(env.size) + targets + PW + 4 + 1
    if policy.startswith("plan"):
        b += L
    if policy == "plan_record":
        b += L * (1 + PW)
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=int, default=1, help="divide the item counts (rehearsal only)")
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    if not torch.cuda.is_available():
        raise SystemExit("playout.py measures on a GPU; none found")
    tmp = tempfile.mkdtemp(prefix="playout_ptxas_")
    procs = start_ptxas(tmp)
    res = {"card": card(), "moves_per_playout": L, "calls": args.calls, "rounds": args.rounds, "rows": []}
    bits4 = torch.arange(4, device="cuda")
    for S, T, W, multi, N, policies, note in ROWS:
        N = max(128, N // args.scale // 128 * 128)
        env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=1)
        g = torch.Generator(device="cuda").manual_seed(2)
        for _ in range(3):      # positions other than the initial ones
            env.raw_move(torch.randint(0, 4, (env.capacity,), dtype=torch.uint8, device="cuda", generator=g))
        PW, cap = env.pos_bytes, env.capacity
        assert cap == N
        plan = torch.randint(0, 4, (L, N), dtype=torch.uint8, device="cuda", generator=g)
        out = (torch.empty(N, PW, dtype=torch.uint8, device="cuda"), torch.empty(N, dtype=torch.int32, device="cuda"),
               torch.empty(N, dtype=torch.uint8, device="cuda"))
        c_out = tuple(torch.empty_like(t) for t in out)
        saved = torch.empty_like(env._pos)
        live = torch.empty(N, dtype=torch.bool, device="cuda")

        def composed(acts, record=False):
            final, steps, won = c_out
            saved.copy_(env._pos)
            final.copy_(env.pos)
            steps.zero_()
            won.zero_()
            live.fill_(True)
            for k in range(L):
                a, ok = acts(k)
                f = env.raw_move(a)
                live.logical_and_(ok)
                steps.add_(live)
                final.copy_(torch.where(live[:, None], env.pos, final))
                if record:
                    c_rec[0][k].copy_(torch.where(live, a, 255))
                    c_rec[1][k].copy_(torch.where(live[:, None], env.pos, 0))
                w = live & ((f & F_WON) != 0)
                won.logical_or_(w)
                live.logical_and_(~w)
            env._pos.copy_(saved)

        def plan_acts(k):
            return plan[k], plan[k] < 4

        def random_acts(k):
            mask = env.valid_moves().long()
            bits = (mask[:, None] >> bits4) & 1
            n = bits.sum(1)
            j = (torch.rand(N, device="cuda") * n).floor().long()
            a = (bits.cumsum(1) <= j[:, None]).sum(1).to(torch.uint8)
            return a, n > 0

        rec = (torch.empty(L, N, dtype=torch.uint8, device="cuda"), torch.empty(L, N, PW, dtype=torch.uint8, device="cuda"))
        c_rec = tuple(torch.empty_like(t) for t in rec) if "plan_record" in policies else None
        for policy in policies:
            if policy == "plan":
                fused = lambda: env.playout(actions=plan, out=out)                                            # noqa: E731
                comp = lambda: composed(plan_acts)                                                             # noqa: E731
            elif policy == "plan_record":
                fused = lambda: env.playout(actions=plan, record=True, out=out + rec)                         # noqa: E731
                comp = lambda: composed(plan_acts, record=True)                                                # noqa: E731
            else:
                fused = lambda: env.playout(n_steps=L, seed=3, out=out)                                       # noqa: E731
                comp = lambda: composed(random_acts)                                                           # noqa: E731
            # same results first
            if policy == "random":
                env.playout(n_steps=L, seed=3, record=True, out=out + rec)
                moves = rec[0]
                check = []

                def replay_acts(k):
                    ok = moves[k] < 4
                    m = env.valid_moves()
                    check.append(bool((((m.long() >> (moves[k].long() & 3)) & 1).bool() | ~ok).all()))
                    return moves[k].contiguous(), ok
                composed(replay_acts)
                # until an item's playout ends the replayed positions are the fused ones: every recorded
                # move is one that valid_moves() allows there
                assert all(check), (S, T)
            else:
                fused()
                comp()
                if policy == "plan_record":
                    assert torch.equal(rec[0], c_rec[0]) and torch.equal(rec[1], c_rec[1]), (S, T)
            assert torch.equal(out[0], c_out[0]) and torch.equal(out[1], c_out[1]) and torch.equal(out[2], c_out[2]), (S, T, policy)
            played = int(out[1].sum())
            fns = {"fused": fused, "composed": comp}
            ms = {k: [] for k in fns}
            for _ in range(args.rounds):
                for k, fn in fns.items():
                    ms[k].append(time_calls(fn, args.calls))
            med = {k: statistics.median(v) for k, v in ms.items()}
            b = item_bytes(env, policy)
            row = {"shape": f"{S}x{S}/{T} tiles/{W} walls {'multi' if multi else 'single'}-colour", "items": N, "policy": policy,
                   "note": note, "kernel": "generic" if T > 8 else ("wide" if S > 8 else "bitboard"), "moves_per_playout": L,
                   "played_moves": played, "won_items": int(out[2].sum()),
                   "algorithmic_bytes_per_item": b, "fused_ms": round(med["fused"], 4), "composed_ms": round(med["composed"], 4),
                   "fused_items_per_s": N / med["fused"] * 1e3, "fused_played_moves_per_s": played / med["fused"] * 1e3,
                   "composed_items_per_s": N / med["composed"] * 1e3, "composed_played_moves_per_s": played / med["composed"] * 1e3,
                   "fused_gb_per_s": round(N * b / med["fused"] / 1e6, 1), "speedup_vs_composed": round(med["composed"] / med["fused"], 2),
                   "rounds_ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}}
            res["rows"].append(row)
            print(json.dumps(row), flush=True)
        del env, plan, out, c_out, saved, live, rec, c_rec
        torch.cuda.empty_cache()
    res["ptxas"] = ptxas_report(procs)
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
