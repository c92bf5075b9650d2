"""Throughput of ts_observe_planes (BatchedTilerSliderEnv.observe_planes) against the HBM write
roofline, beside what a user pays today for the same planes.

  python profiles/experiments/observe_planes.py --out /tmp/observe_planes.json

Shapes (every output larger than the 126 MB L2): 6x6 / 4 tiles / 8 walls multi-colour and 5x5 /
1 tile / 5 walls single-colour at 4,194,304 envs, 12x12 / 8 tiles / 36 walls multi-colour at
1,048,576 envs; synthetic() puzzles (distinct target cells), each in uint8, bfloat16, float16 and
float32.  Per row, on the same batch in the same run:
  planes    observe_planes(out) into a preallocated [N, C, S, S] tensor;
  observe   (a) observe(obs) into a preallocated float32 [N, S, S, 3] tensor;
  torch     (b) observe(obs) followed by the cheapest PyTorch composition of the same planes in
            the same dtype from it: single colour one cast-and-transpose copy; multi colour one
            copy of the wall channel and one broadcast compare of the tile channel against 1..T
            and of the target channel against 1..NT, each stored into its planes of a
            preallocated output (the compare is exact only for distinct targets, which these
            puzzles have).  Its result is checked equal to observe_planes() before timing.
Timing: CUDA events around `--calls` back-to-back calls after 3 warm-up calls, `--rounds` rounds
alternating the three; the median round is reported.  GB/s counts the bytes of the planes tensor
(what the kernel must write); the fraction is of the 6,534.1 GB/s copy bandwidth measured on a
B200 (SURVEY.md).
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

COPY_GBPS = 6534.1
SHAPES = [(6, 4, 8, True, 4_194_304), (5, 1, 5, False, 4_194_304), (12, 8, 36, True, 1_048_576)]


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock_sm_clock": q[0] if q else None}


def torch_planes(env, obs, out):
    """(b): the planes from observe()'s float32 [N, S, S, 3] in PyTorch."""
    import torch
    if env.goal_mode != 0:
        out.copy_(obs.permute(0, 3, 1, 2))
        return out
    T, C = env.n_tiles, out.shape[1]
    out[:, 0].copy_(obs[..., 0])
    if T:
        out[:, 1:1 + T].copy_((obs[..., 1:2] == torch.arange(1, T + 1, device=obs.device, dtype=obs.dtype)).permute(0, 3, 1, 2))
    if C > 1 + T:
        out[:, 1 + T:].copy_((obs[..., 2:3] == torch.arange(1, C - T, device=obs.device, dtype=obs.dtype)).permute(0, 3, 1, 2))
    return out


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=int, default=1, help="divide the env counts (rehearsal only)")
    args = ap.parse_args()
    import torch
    import tiler_slider_b200 as ts
    if not torch.cuda.is_available():
        raise SystemExit("observe_planes.py measures on a GPU; none found")
    res = {"card": card(), "copy_gbps": COPY_GBPS, "calls": args.calls, "rounds": args.rounds, "rows": []}
    for S, T, W, multi, N in SHAPES:
        N //= args.scale
        env = ts.BatchedTilerSliderEnv.synthetic(N, S, T, W, multi, seed=1)
        C = env.plane_count
        obs = torch.empty(N, S, S, 3, dtype=torch.float32, device="cuda")
        for dtype in (torch.uint8, torch.bfloat16, torch.float16, torch.float32):
            out = torch.empty(N, C, S, S, dtype=dtype, device="cuda")
            ref = torch.empty_like(out)
            env.observe_planes(out, dtype=dtype)
            torch_planes(env, env.observe(obs), ref)
            assert torch.equal(out, ref), (S, T, dtype)
            del ref
            fns = {"planes": lambda: env.observe_planes(out, dtype=dtype),
                   "observe": lambda: env.observe(obs),
                   "torch": lambda: torch_planes(env, env.observe(obs), out)}
            ms = {k: [] for k in fns}
            for _ in range(args.rounds):
                for k, fn in fns.items():
                    ms[k].append(time_calls(fn, args.calls))
            med = {k: statistics.median(v) for k, v in ms.items()}
            gb = out.numel() * out.element_size() / 1e9
            row = {"shape": f"{S}x{S}/{T} tiles/{W} walls {'multi' if multi else 'single'}-colour", "n_envs": N,
                   "dtype": str(dtype).replace("torch.", ""), "channels": C, "bytes_per_env": C * S * S * out.element_size(),
                   "planes_ms": round(med["planes"], 4), "planes_gb_written_per_s": round(gb / med["planes"] * 1e3, 1),
                   "planes_obs_per_s": N / med["planes"] * 1e3,
                   "planes_fraction_of_copy_bw": round(gb / med["planes"] * 1e3 / COPY_GBPS, 3),
                   "observe_ms": round(med["observe"], 4), "observe_then_torch_ms": round(med["torch"], 4),
                   "speedup_vs_observe_then_torch": round(med["torch"] / med["planes"], 2),
                   "rounds_ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}}
            res["rows"].append(row)
            print(json.dumps(row), flush=True)
            del out
        del env, obs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
