"""bench.py -- env-steps/s of the Tiler-Slider step path on B200, with its HBM roofline and the
CPU step loop beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[2], the one its metric is quoted on): 6x6 boards, 4
coloured tiles and targets (ordered goal), 8 random walls, 16,777,216 envs PER GPU (weak scaling:
envs are independent, sharded by index, no collective on the step path), uniform random actions,
max_steps=100, auto-reset on.  A "step" is one ts_step launch advancing every env by one action.

How a number is taken (DESIGN.md section 6):
  * a block of K steps is replayed from CUDA graphs of up to 50 ts_step launches each (one
    launch per step); after the W warm-up steps blocks are replayed until the GPU has been busy
    for >= 150 ms, so the graphs are resident and the SM clock has left its idle state before
    anything is timed (the round-1 line timed 1.5 ms straight after start-up and read 2x slow on
    8 GPUs);
  * the batch is then reset to its initial boards, whole blocks of at least 256 steps in all
    run untimed back to back, and exactly K steps are timed right behind them with CUDA events
    on the launching stream, so that they run under continuous load and are queued before the
    GPU reaches them; the job time is the MAX over ranks, and the line carries first / best /
    worst graph chunk and per-rank [min, median, max] so that a straggler is visible instead of
    folded into the headline;
  * what those K steps compute depends only on the arguments: the same puzzles, action rows and
    start state on every run, so `--dump-outputs DIR` can store the last step's outputs for
    comparing two builds;
  * NVML clocks / throttle reasons are read by the main thread every 0.5 ms while the GPU works
    through the untimed and the timed steps (no polling thread competing with the launches).
`value` = total env-steps/s over all ranks with actions resident in HBM.  `e2e` = the same step
driven from pinned HOST buffers through ts_step_host (actions uploaded, reward+done downloaded
every step).  `roofline` = algorithmic bytes (3T + ceil(S^2/8) + 8 per env-step, SURVEY 8(d)) over
the measured launch duration, against MEASURED_PEAKS.json.  `configs` = the other BASELINE configs
(c2, c4, c5 = BFS), each with its own roofline and parity count.  `cpu_baseline` = the reference's
Python step loop restated in oracle/py_port.py, timed on this box's host cores (the reference is
pure Python and is not on this box).  `--impl reference` times that loop on all host cores.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import time
from dataclasses import dataclass

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


@dataclass(frozen=True)
class Config:
    name: str
    size: int
    tiles: int
    walls: int
    multi: bool
    envs: int            # per GPU (weak) / in total (strong)
    puzzle_seed: int
    action_seed: int

    @property
    def algo_bytes(self) -> int:          # SURVEY 8(d): 3T + ceil(S^2/8) + 8
        return 3 * self.tiles + (self.size * self.size + 7) // 8 + 8


# BASELINE.json configs (SURVEY 8(d) table): c3 is the one the metric is quoted on
CONFIGS = {"c2": Config("c2", 5, 1, 5, False, 1_048_576, 1001, 2001),
           "c3": Config("c3", 6, 4, 8, True, 16_777_216, 1002, 2002),
           "c4": Config("c4", 12, 8, 36, True, 4_194_304, 1003, 2003)}
MAX_STEPS = 100
METRIC = "env-steps/sec at 1/2/4/8 B200 and % HBM roofline vs reference CPU step loop"
UNIT = "env-steps/s"
N_ACTION_ROWS = 8                               # distinct pre-generated action vectors, cycled
GRAPH_STEPS_MAX = 50                            # launches per captured graph
RAMP_MS = 150.0                                 # GPU-busy time before the timed steps
PREROLL_STEPS = 256                             # untimed steps right before the timed ones (whole blocks)
L2_BYTES = 126e6
DUMP_BYTES = 60_000_000                         # --dump-outputs: array bytes written, at most


def bytes_moved(cfg: Config, ts) -> dict:
    """Bytes the step kernel's loads and stores request per env-step in the auto-reset fast path
    (no status byte): what has to cross HBM when nothing is cached between steps."""
    lib = ts.lib()
    pw = lib.ts_pos_bytes(cfg.tiles)
    walls = lib.ts_walls_bytes(cfg.size) // (2 if cfg.size > 8 else 1)     # wide boards: one of the two axis records
    tg = pw if (cfg.multi or cfg.tiles == 1) else lib.ts_target_board_bytes(cfg.size)
    rd, wr = pw + walls + tg + 1 + 1, pw + 1 + 4 + 1
    return {"read": rd, "written": wr, "total": rd + wr}


def workload_config(cfg: Config, n_gpus: int, envs_per_gpu: int, extra: dict | None = None) -> dict:
    S, T = cfg.size, cfg.tiles
    ws = envs_per_gpu * cfg.algo_bytes
    out = {"workload": f"{cfg.name}: {S}x{S} boards, {T} {'coloured ' if cfg.multi else ''}tile(s)+target(s) "
                       f"({'ordered' if cfg.multi else 'set'} goal), {cfg.walls} walls, {envs_per_gpu} envs per GPU "
                       f"sharded by index over {n_gpus} GPU(s), uniform random actions, max_steps={MAX_STEPS}, auto-reset",
           "size": S, "tiles": T, "walls": cfg.walls, "multi_color": cfg.multi, "envs_per_gpu": envs_per_gpu,
           "envs_total": envs_per_gpu * n_gpus, "max_steps": MAX_STEPS, "auto_reset": True,
           "outputs": "next state (packed positions), reward f32, done u8 per env-step (status byte not stored: track_flags=False)",
           "algorithmic_bytes_per_env_step": cfg.algo_bytes,
           "l2_policy": (f"inputs larger than L2 ({ws / 1e6:.0f} MB of algorithmic state+io per step vs 126 MB L2); no flush needed"
                         if ws > L2_BYTES else
                         f"working set {ws / 1e6:.0f} MB per step fits the 126 MB L2: steps run L2-resident (stated, not flushed)"),
           "parallelism": f"env-index sharding x{n_gpus}, no collective on the step path"}
    if extra:
        out.update(extra)
    return out


def dump_outputs(env, out_dir: str) -> None:
    """What the last step returned to its caller -- state (as tile positions), reward, done -- as
    float32 .npy files in out_dir, with the float64 indices of the envs they belong to.  Above
    DUMP_BYTES the envs are a fixed, seeded sample, the same for every build and run."""
    import numpy as np
    import torch
    n = env.n_envs
    m = min(n, DUMP_BYTES // (4 * (2 * env.n_tiles + 2) + 8))
    idx = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    sel = torch.from_numpy(idx).to(env.device)
    arrays = {"env_index": idx.astype(np.float64), "positions": env.positions()[sel].float().cpu().numpy(),
              "reward": env.reward[sel].cpu().numpy(), "done": env.done[sel].float().cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """One process: its own envs, W warm-up + K timed passes of the reference-style loop."""
    puzzles, actions, warmup, steps = args
    from oracle import py_port
    envs = [py_port.PortEnv(s, b, i, t, m, MAX_STEPS) for (s, b, i, t, m) in puzzles]
    for e in envs:
        e.reset()

    def one_pass(k):
        row = actions[k % len(actions)]
        for j, e in enumerate(envs):
            _, done, _ = e.step(int(row[j]))
            if done:
                e.reset()
    for k in range(warmup):
        one_pass(k)
    t0 = time.perf_counter()
    for k in range(steps):
        one_pass(warmup + k)
    return time.perf_counter() - t0, len(envs) * steps


def synth_puzzles_host(cfg: Config, n: int, seed: int):
    """Host copy of the synthetic recipe (random permutation prefix; environment.py:221-226)
    for the CPU legs, which must not need a GPU."""
    import numpy as np
    S, T, W = cfg.size, cfg.tiles, cfg.walls
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        perm = rng.permutation(S * S)
        cells = [(int(c) // S, int(c) % S) for c in perm]
        out.append((S, cells[:W], cells[W:W + T], cells[W + T:W + 2 * T], cfg.multi))
    return out


def cpu_loop_rate(cfg: Config, n_procs: int, steps: int, warmup: int, budget_s: float):
    """env-steps/s of the Python step loop on n_procs processes, sized to ~budget_s."""
    import numpy as np
    est_rate = 3.0e4                                   # per core, SURVEY section 6
    envs_per_proc = int(max(1, min(4096, budget_s * est_rate / max(1, steps + warmup))))
    rng = np.random.default_rng(cfg.action_seed)
    jobs = []
    for p in range(n_procs):
        acts = rng.integers(0, 4, size=(min(steps + warmup, 256), envs_per_proc), dtype=np.uint8)
        jobs.append((synth_puzzles_host(cfg, envs_per_proc, cfg.puzzle_seed + p), acts, warmup, steps))
    if n_procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(n_procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    elapsed = max(r[0] for r in res)
    total = sum(r[1] for r in res)
    return total / elapsed, elapsed, envs_per_proc


def c_oracle_rate(cfg: Config, n_envs: int = 4096, steps: int = 200):
    import numpy as np
    from oracle import oracle as orc
    S, T, W = cfg.size, cfg.tiles, cfg.walls
    rng = np.random.default_rng(cfg.puzzle_seed)
    perm = np.argsort(rng.random((n_envs, S * S)), axis=1)
    blocked = np.zeros((n_envs, S * S), np.uint8)
    np.put_along_axis(blocked, perm[:, :W], 1, axis=1)
    tc, gc = perm[:, W:W + T], perm[:, W + T:W + 2 * T]
    tiles = np.stack([tc // S, tc % S], -1).astype(np.uint8)
    targets = np.stack([gc // S, gc % S], -1).astype(np.uint8)
    actions = rng.integers(0, 4, size=(steps, n_envs), dtype=np.uint8)
    t0 = time.perf_counter()
    orc.rollout(S, cfg.multi, blocked, tiles, targets, actions, max_steps=MAX_STEPS, auto_reset=True)
    return n_envs * steps / (time.perf_counter() - t0)


def parity_check(ts, dev, cfg: Config, n_envs: int = 8192, steps: int = 128) -> dict:
    """The parity run that accompanies a throughput number (SURVEY 8(d)): the first n_envs
    puzzles of the bench workload, `steps` random actions, every position / flag / reward of the
    CUDA path compared with the C oracle (the checker, part of the cpu_baseline leg); the same
    batch is also stepped in the bench's fast path (no status byte) and must agree."""
    import numpy as np
    import torch
    from oracle import oracle as orc
    S, T, W, multi = cfg.size, cfg.tiles, cfg.walls, cfg.multi
    kw = dict(seed=cfg.puzzle_seed, max_steps=MAX_STEPS, auto_reset=True, track_terminal=True, device=dev)
    env = ts.BatchedTilerSliderEnv.synthetic(n_envs, S, T, W, multi, **kw)
    fast = ts.BatchedTilerSliderEnv.synthetic(n_envs, S, T, W, multi, track_flags=False, **kw)
    blocked = env.blocked_cells().cpu().numpy().astype(np.uint8)
    tiles = env.positions().cpu().numpy()
    if env.goal_mode == ts.GOAL_ORDERED:
        targets = env.target_positions().cpu().numpy()
    else:
        cells = np.stack([np.flatnonzero(r) for r in env.target_positions().cpu().numpy()])
        targets = np.stack([cells // S, cells % S], -1).astype(np.uint8)
    gen = torch.Generator(device=dev).manual_seed(cfg.action_seed)
    actions = torch.randint(0, 4, (steps, env.capacity), dtype=torch.uint8, device=dev, generator=gen)
    want = orc.rollout(S, multi, blocked, tiles, targets, actions[:, :n_envs].cpu().numpy(), max_steps=MAX_STEPS, auto_reset=True)
    bad = fast_bad = 0
    for k in range(steps):
        count_before = env.step_count.to(torch.int32).cpu().numpy()      # info['step_count'] is pre-increment (environment.py:128)
        _, r, d = env.step(actions[k])
        post = torch.where(d[:, None, None], env.positions(env.terminal_pos), env.positions())
        bad += int((post.cpu().numpy() != want["pos"][k]).any(axis=(1, 2)).sum())
        bad += int((env.flags.cpu().numpy() != want["flags"][k]).sum())
        bad += int((r.cpu().numpy() != want["reward"][k]).sum())
        bad += int((count_before != want["count"][k]).sum())
        _, rf, df = fast.step(actions[k])
        fast_bad += int(not torch.equal(fast.pos, env.pos)) + int(not torch.equal(rf, r)) + int(not torch.equal(df, d))
    # K3 / valid-move mask of the states the rollout ended in (first n_obs envs), against the oracle
    n_obs = min(n_envs, 1024)
    obs = env.observe()[:n_obs].cpu().numpy()
    valid = env.valid_moves()[:n_obs].cpu().numpy()
    blocked_rc = [np.argwhere(b.reshape(S, S)) for b in blocked[:n_obs]]
    obs_bad = 0
    for i in range(n_obs):
        st = orc.OracleState(S, blocked_rc[i], want["final_pos"][i], targets[i], multi)
        obs_bad += int((st.get_state_array() != obs[i]).any())
        obs_bad += int(sum(1 << d for d in st.valid_moves()) != int(valid[i]))
    return {"env_steps_checked": n_envs * steps, "mismatches": bad, "fast_path_mismatches": fast_bad,
            "fields": "positions per tile, flags (done/won/invalid/timeout), reward, pre-increment step_count",
            "observations_checked": n_obs, "observation_or_valid_mask_mismatches": obs_bad,
            "checker": "oracle/ts_oracle.c"}


def run_reference(args) -> int:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    rate, elapsed, envs_per_proc = cpu_loop_rate(cfg, cores, args.steps, args.warmup, budget_s=25.0)
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / max(1, args.steps),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": workload_config(cfg, args.gpus, args.envs),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{cores} processes x {envs_per_proc} envs x {args.steps} steps of the same "
                                       f"{cfg.size}x{cfg.size}/{cfg.tiles}-tile workload; oracle/py_port.py = the reference's "
                                       "Python step loop restated (the pure-Python reference cannot travel to this box)"},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------
# clocks (NVML, read by the main thread while the GPU works through the queued blocks)
# ------------------------------------------------------------------------------------------
class Clocks:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting",
               0x10: "sync_boost"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self.nv = [], set(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for b, name in self.REASONS.items():
                if bits & b:
                    self.reasons.add(name)
        except Exception:
            pass

    def sample_until(self, event, period_s: float = 0.0005, limit_s: float = 30.0):
        t0 = time.perf_counter()
        while not event.query() and time.perf_counter() - t0 < limit_s:
            self.sample()
            time.sleep(period_s)

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_min_mhz": s[0] if s else None, "sm_max_mhz": self.max_mhz,
                "samples": len(s), "reasons": sorted(self.reasons),
                "how": "NVML, main thread, while the GPU executes the untimed steps before the timed ones and the timed ones"}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
class Runner:
    def __init__(self):
        import torch
        import torch.distributed as dist
        import tiler_slider_b200 as ts
        self.torch, self.dist, self.ts = torch, dist, ts
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                self.peaks = json.load(f)
        except Exception:
            pass
        self.peak = float(self.peaks.get("hbm_gbs", 6650.0))
        self.peak_source = "MEASURED_PEAKS.json hbm_gbs (of measured)" if self.peaks else "fallback 6650 GB/s (of fallback)"

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def gather(self, values):
        """[world][len(values)] float64 list of every rank's values."""
        torch = self.torch
        mine = torch.tensor(values, dtype=torch.float64, device=self.dev)
        if self.world == 1:
            return [mine.tolist()]
        out = torch.empty(self.world * mine.numel(), dtype=torch.float64, device=self.dev)
        self.dist.all_gather_into_tensor(out, mine)
        return out.view(self.world, -1).tolist()

    def measure(self, cfg: Config, n_local: int, steps: int, warmup: int, use_graph: bool = True,
                clocks: Clocks | None = None, ramp_ms: float = RAMP_MS, dump_dir: str | None = None) -> dict:
        """Device-resident throughput of one config (see the module docstring)."""
        torch, ts = self.torch, self.ts
        env = ts.BatchedTilerSliderEnv.synthetic(n_local, cfg.size, cfg.tiles, cfg.walls, cfg.multi, seed=cfg.puzzle_seed,
                                                 env_index_base=self.rank * n_local, max_steps=MAX_STEPS, auto_reset=True,
                                                 track_flags=False, device=self.dev)
        gen = torch.Generator(device=self.dev).manual_seed(cfg.action_seed + self.rank)
        actions = torch.randint(0, 4, (N_ACTION_ROWS, env.capacity), dtype=torch.uint8, device=self.dev, generator=gen)
        for k in range(warmup):                                   # the W warm-up steps, launched one by one
            env.step(actions[k % N_ACTION_ROWS])
        # a block is `steps` steps in chunks of at most GRAPH_STEPS_MAX; step k of a chunk takes action row k
        cs = min(steps, GRAPH_STEPS_MAX)
        n_rep, rem = divmod(steps, cs)
        chunks = [cs] * n_rep + ([rem] if rem else [])
        if use_graph:
            rows = actions[torch.arange(cs, device=self.dev) % N_ACTION_ROWS] if cs > N_ACTION_ROWS else actions[:cs]
            graphs = {cs: env.capture_steps(rows.contiguous())}
            if rem:
                graphs[rem] = env.capture_steps(rows[:rem].contiguous())

            def chunk(n):
                graphs[n].replay()
        else:
            def chunk(n):
                for k in range(n):
                    env.step(actions[k % N_ACTION_ROWS])

        def block():
            for n in chunks:
                chunk(n)
        # graph upload + clock ramp: keep the GPU busy for RAMP_MS before anything is timed
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        block()
        torch.cuda.synchronize()
        ramp_blocks, busy_ms = 1, 0.0
        while ramp_blocks == 1 or busy_ms < ramp_ms:
            ev0.record()
            block()
            ev1.record()
            ev1.synchronize()
            busy_ms += ev0.elapsed_time(ev1)
            ramp_blocks += 1
        self.barrier()
        # back to the initial boards, so that what the timed steps compute does not depend on how long
        # the ramp ran; then untimed blocks back to back, so that the timed steps run under continuous
        # load as they would in a long run
        env.reset()
        pre_blocks = -(-PREROLL_STEPS // steps)
        for _ in range(pre_blocks):
            block()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(len(chunks) + 1)]
        marks[0].record()
        for i, n in enumerate(chunks):                            # exactly `steps` timed launches, back to back
            chunk(n)
            marks[i + 1].record()
        if clocks is not None:          # from the untimed steps on: a throttle they bring on shows too
            clocks.sample_until(marks[-1])
        self.barrier()
        if dump_dir is not None and self.rank == 0:
            dump_outputs(env, dump_dir)
        mine = [marks[i].elapsed_time(marks[i + 1]) / n for i, n in enumerate(chunks)] + [marks[0].elapsed_time(marks[-1])]
        per_rank = self.gather(mine)                              # [world][chunks + 1]: ms per step of each chunk, total ms
        total = max(r[-1] for r in per_rank)
        per_chunk = [max(r[i] for r in per_rank) for i in range(len(chunks))]
        total_envs = n_local * self.world
        per_launch_s = total * 1e-3 / steps
        achieved = cfg.algo_bytes * n_local / per_launch_s / 1e9
        moved = bytes_moved(cfg, ts)
        wins = int(self.gather([float(env.is_won().sum())])[0][0]) if self.world == 1 else \
            int(sum(r[0] for r in self.gather([float(env.is_won().sum())])))
        kernel = f"ts::step_kernel<{cfg.size},{cfg.tiles}>" if cfg.size <= 8 else f"ts::wide_step_kernel<{cfg.tiles}>"
        out = {"value": total_envs * steps / (total * 1e-3), "ms_per_step": total / steps,
               "blocks": {"n": len(chunks), "steps_per_block": cs,
                          "statistic": "value: all timed steps back to back (max over ranks); first / best / worst and "
                                       "per rank: per graph chunk of up to 50 of them",
                          "first_ms_per_step": per_chunk[0], "best_ms_per_step": min(per_chunk),
                          "worst_ms_per_step": max(per_chunk),
                          "per_rank_ms_per_step_min_med_max": [[min(r[:-1]), sorted(r[:-1])[len(chunks) // 2], max(r[:-1])]
                                                               for r in per_rank]},
               "warmup_launches": warmup + (ramp_blocks + pre_blocks) * steps,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak,
                            "traffic": None, "kernel": kernel,
                            "algorithmic_bytes_per_launch": cfg.algo_bytes * n_local, "avg_launch_ms": per_launch_s * 1e3,
                            "bytes_moved_per_env_step": moved,
                            "frac_on_bytes_moved": moved["total"] * n_local / per_launch_s / 1e9 / self.peak,
                            "per_rank_frac": [cfg.algo_bytes * n_local / (r[-1] * 1e-3 / steps) / 1e9 / self.peak
                                              for r in per_rank],
                            "peak_source": self.peak_source},
               "gpu_launches": steps, "wins_in_last_step": wins, "cuda_graph": bool(use_graph),
               "envs_per_gpu": n_local}
        traffic = ncu_traffic(cfg, n_local)
        if traffic:
            out["roofline"]["traffic"] = traffic["dram_bytes_per_launch"]
            out["roofline"]["traffic_source"] = traffic["source"]
        return out

    # ---- end to end through host buffers -----------------------------------------------------
    def e2e(self, cfg: Config, n_local: int, steps: int) -> dict:
        torch, ts = self.torch, self.ts
        env = ts.BatchedTilerSliderEnv.synthetic(n_local, cfg.size, cfg.tiles, cfg.walls, cfg.multi, seed=cfg.puzzle_seed,
                                                 env_index_base=self.rank * n_local, max_steps=MAX_STEPS, auto_reset=True,
                                                 device=self.dev)
        h_act = torch.randint(0, 4, (n_local,), dtype=torch.uint8).pin_memory()
        h_rew = torch.empty(n_local, dtype=torch.float32).pin_memory()
        h_done = torch.empty(n_local, dtype=torch.uint8).pin_memory()
        h_flags = torch.empty(n_local, dtype=torch.uint8).pin_memory()

        def timed(fn, n_warm):
            for _ in range(n_warm):
                fn()
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()                                   # returns after the results landed on the host
            self.barrier()
            secs = max(r[0] for r in self.gather([time.perf_counter() - t0]))
            return n_local * self.world * steps / secs
        full = timed(lambda: env.step_host(h_act, h_rew, h_done), 3)
        compact = timed(lambda: env.step_host(h_act, h_flags=h_flags), 2)
        tot = n_local * self.world
        return {"value": full, "unit": UNIT, "h2d_bytes_per_step": tot, "d2h_bytes_per_step": 5 * tot, "steps": steps,
                "path": "BatchedTilerSliderEnv.step_host -> ts_step_host (pinned host actions in, reward f32 + done u8 out)",
                "compact_variant": {"value": compact, "d2h_bytes_per_step": tot,
                                    "what": "same call, only the 1-byte status word downloaded (done = bit 0, "
                                            "reward = function of the WON / INVALID bits)"}}

    # ---- BASELINE config 5: batched BFS ---------------------------------------------------------
    def bfs(self, puzzles_per_gpu: int, n_check: int) -> dict:
        import numpy as np
        torch, ts, dist = self.torch, self.ts, self.dist
        from tiler_slider_b200.bfs import BfsSolver
        S, T, W, seed = 6, 4, 8, 1004
        P = puzzles_per_gpu * self.world
        table = ts.BatchedTilerSliderEnv.synthetic(P, S, T, W, True, seed=seed, device=self.dev)
        out = {"workload": f"c5: BFS to exhaustion over {P} synthetic {S}x{S} puzzles, {T} coloured tiles, {W} walls "
                           f"({puzzles_per_gpu} per GPU), key = puzzle id || positions",
               "unit": "generated successors/s (state x move)", "n_gpus": self.world, "puzzles": P}

        def run(solver, **kw):
            times, res = [], None
            for _ in range(2):                         # the first search also pays the allocations (cold)
                self.barrier()
                t0 = time.perf_counter()
                res = solver.solve(**kw)
                self.barrier()
                times.append(max(r[0] for r in self.gather([time.perf_counter() - t0])))
            return res, times

        if self.world > 1:   # create the NCCL channels outside the timed region
            w = torch.zeros(self.world, dtype=torch.int64, device=self.dev)
            dist.all_to_all_single(torch.empty_like(w), w)
            dist.all_reduce(w)
        BfsSolver(ts.BatchedTilerSliderEnv.synthetic(128, S, T, W, True, seed=1, device=self.dev),
                  table_capacity=1 << 22, exchange="nccl").solve(max_depth=3)          # warm the kernels / allocator
        log2 = max(16, int(np.ceil(np.log2(P * 16384 / self.world))))      # ~3,400 states per puzzle on average
        results = {}
        solver = BfsSolver(table, table_capacity=1 << log2, exchange="auto")
        res, (cold, warm) = run(solver)
        results["hash"] = res
        # algorithmic bytes per successor of the hash-partitioned path: SURVEY 8(d), ~42 B of HBM traffic
        out["hash_partitioned"] = {
            "value": res.generated / warm, "seconds": warm, "seconds_cold": cold, "unique_states": res.n_states,
            "generated_successors": res.generated, "depth": len(res.levels) - 1, "table_log2_per_rank": log2,
            "exchange": (solver.exchange if self.world > 1 else "none (one rank)"),
            # keys that crossed NVLink: 8 bytes each, (G-1)/G of the keys a rank sends have a remote owner
            "nvlink": ({"keys_exchanged": res.exchanged_keys,
                        "bytes_per_gpu_per_direction": 8 * res.exchanged_keys * (self.world - 1) / self.world / self.world,
                        "GBps_per_gpu_per_direction": 8 * res.exchanged_keys * (self.world - 1) / self.world / self.world / warm / 1e9,
                        "of_measured_peer_copy_770_GBps": 8 * res.exchanged_keys * (self.world - 1) / self.world / self.world / warm / 1e9 / 770.0}
                       if self.world > 1 and res.exchanged_keys else None),
            "roofline": {"bound": "hbm", "achieved": 42 * res.generated / self.world / warm / 1e9, "peak": self.peak, "unit": "GB/s",
                         "frac": 42 * res.generated / self.world / warm / 1e9 / self.peak, "traffic": None,
                         "kernel": "ts::bfs_hash_insert_kernel (K5) + bfs_expand(_exchange)_kernel (K4/K4x)",
                         "algorithmic_bytes_per_successor": 42, "peak_source": self.peak_source}}
        del solver
        torch.cuda.empty_cache()
        from tiler_slider_b200.bfs import LocalBfs
        local = LocalBfs(table)
        resl, (coldl, warml) = run(local)
        results["local"] = resl
        out["per_puzzle_on_chip"] = {
            "value": resl.generated / warml, "seconds": warml, "seconds_cold": coldl, "unique_states": resl.n_states,
            "generated_successors": resl.generated, "depth": len(resl.levels) - 1,
            "what": "K6: one CTA per puzzle, visited set = perfect-hash bitmap in shared memory, live levels in a shared-memory "
                    "ring (spilling to HBM), puzzles sharded over the ranks with no exchange",
            "plan_rank0": local.plan(), "fallback_puzzles": int(resl.fallback_puzzles),
            "roofline": {"bound": "on-chip (instruction issue / shared-memory latency); the 42 B per successor of SURVEY 8(d) are not moved",
                         "hbm_equivalent_GBps": 42 * resl.generated / self.world / warml / 1e9,
                         "dram_bytes_per_search_ncu": "about 1 MB per 65,536 puzzles (profiles/r2_ncu_bfs_local_raw.csv)"}}
        out["value"] = max(v["value"] for k, v in out.items() if isinstance(v, dict) and "value" in v)
        # per-puzzle results against the CPU oracle's BFS (rank 0)
        ok, n_chk = True, 0
        if self.rank == 0 and n_check:
            from oracle import oracle as orc
            blocked = table.blocked_cells()[:n_check].cpu().numpy()
            tiles = table.positions()[:n_check].cpu().numpy()
            targets = table.target_positions()[:n_check].cpu().numpy()
            n_chk = min(n_check, P)
            t0 = time.perf_counter()
            for e in range(n_chk):
                b = [(c // S, c % S) for c in np.flatnonzero(blocked[e])]
                n, _, depth, _ = orc.OracleState(S, b, tiles[e].tolist(), targets[e].tolist(), True).bfs(max_states=1 << 22)
                for r in results.values():
                    ok &= n == int(r.states_per_puzzle[e]) and depth == int(r.solve_depth_per_puzzle[e])
            out["oracle_seconds"] = time.perf_counter() - t0
        if len(results) == 2:      # the two GPU searches agree on every puzzle
            a, b = results["hash"], results["local"]
            ok &= bool(torch.equal(a.states_per_puzzle, b.states_per_puzzle)) and \
                bool(torch.equal(a.solve_depth_per_puzzle.to(torch.int64), b.solve_depth_per_puzzle.to(torch.int64))) and a.levels == b.levels
        out["oracle_check"] = {"puzzles": n_chk, "ok": bool(ok), "checker": "oracle/ts_oracle.c tso_bfs (states per puzzle, solve depth)",
                               "gpu_paths_agree_on_all_puzzles": len(results) == 2}
        return out

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def ncu_traffic(cfg: Config, n_local: int) -> dict | None:
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the config's step kernel from the
    committed ncu capture of this round (profiles/r2_traffic.json, written from the ncu pages next to
    it), valid for the env count it was captured at."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            t = json.load(f).get(cfg.name)
        if t and int(t["envs"]) == n_local:
            return t
    except Exception:
        pass
    return None


def run_ours(args) -> int:
    # stdout carries exactly ONE line, the JSON: libraries that print to fd 1 (NCCL's version banner
    # when a communicator is created) are sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    R = Runner()
    cfg = CONFIGS[args.config]
    n_local = args.envs
    clk = Clocks(R.local)
    head = R.measure(cfg, n_local, args.steps, args.warmup, use_graph=args.graph, clocks=clk, ramp_ms=args.ramp_ms,
                     dump_dir=args.dump_outputs)
    clocks = clk.summary()
    e2e = R.e2e(cfg, n_local, max(3, min(args.steps, args.e2e_steps))) if args.e2e_steps > 0 else None
    line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": R.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(cfg, R.world, n_local),
            "roofline": head["roofline"], "e2e": e2e, "gpu_launches": head["gpu_launches"], "clocks": clocks,
            "cuda_graph": head["cuda_graph"], "blocks": head["blocks"], "warmup_launches": head["warmup_launches"],
            "wins_in_last_step": head["wins_in_last_step"]}
    if not args.no_extra:
        extra = {}
        # BASELINE's literal "16M envs sharded over 1/2/4/8": the config's env count split over the ranks
        if R.world > 1 and args.scaling == "weak":
            n_strong = -(-cfg.envs // R.world)
            s = R.measure(cfg, n_strong, args.steps, 3)
            line["strong_scaling"] = {"envs_total": n_strong * R.world, "envs_per_gpu": n_strong, "value": s["value"],
                                      "ms_per_step": s["ms_per_step"], "roofline_frac": s["roofline"]["frac"], "blocks": s["blocks"]}
        for name in ("c2", "c3", "c4"):
            if name == args.config:
                continue
            c = CONFIGS[name]
            m = R.measure(c, c.envs, args.steps, 3)
            extra[name] = {"value": m["value"], "unit": UNIT, "ms_per_step": m["ms_per_step"],
                           "config": workload_config(c, R.world, c.envs), "roofline": m["roofline"], "blocks": m["blocks"],
                           "gpu_launches": m["gpu_launches"]}
            if R.rank == 0 and not args.no_cpu:
                extra[name]["parity"] = parity_check(R.ts, R.dev, c)
            R.torch.cuda.empty_cache()
        R.barrier()
        extra["c5"] = R.bfs(args.bfs_puzzles, 0 if args.no_cpu else args.bfs_check)
        line["configs"] = extra
    if R.rank == 0:
        if not args.no_cpu:
            line["parity"] = parity_check(R.ts, R.dev, cfg)
            if R.world == 1:
                rate, elapsed, n_cpu = cpu_loop_rate(cfg, 1, 300, 10, budget_s=12.0)
                line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                                        "sample": f"{n_cpu} envs x 300 steps of the same workload, single process, "
                                                  "oracle/py_port.py (reference Python step loop restated)",
                                        "c_oracle_env_steps_per_s_1core": c_oracle_rate(cfg)}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    R.barrier()
    R.close()
    return 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c3")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the config's)")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak (default): the config's env count on EVERY GPU; strong: that count split over the GPUs")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU legs (cpu_baseline, oracle parity checks)")
    ap.add_argument("--no-extra", action="store_true", help="headline config only (no `configs`, no strong-scaling figure)")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch every step from Python instead of replaying CUDA graphs")
    ap.add_argument("--ramp-ms", type=float, default=RAMP_MS, help="GPU-busy time before the timed steps (profiling runs: 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the headline config returned "
                    "(a fixed sample of envs) to DIR/<name>.npy, to compare two builds output for output")
    ap.add_argument("--bfs-puzzles", type=int, default=65_536, help="c5: puzzles per GPU")
    ap.add_argument("--bfs-check", type=int, default=1024, help="c5: puzzles cross-checked against the CPU oracle's BFS")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.envs is None:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        args.envs = cfg.envs if args.scaling == "weak" else -(-cfg.envs // world)
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
