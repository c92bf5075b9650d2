"""Regenerate the measured tables of README.md and DESIGN.md from the kept bench lines
(profiles/r8_bench_n1.json for one GPU, profiles/r2_bench_n{2,4,8}.json for several), between the
<!-- BEGIN/END ... --> markers, so that every number in the docs is a number of an artifact:
    python profiles/experiments/make_tables.py"""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def f(x):
    return f"{x:.2e}".replace("e+", "e")


def load():
    out = {}
    # one GPU: the step with alternating traversal order (round 8); several GPUs: round 2's lines
    for n, name in ((1, "r8_bench_n1.json"), (2, "r2_bench_n2.json"), (4, "r2_bench_n4.json"), (8, "r2_bench_n8.json")):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            with open(p) as fh:
                out[n] = json.loads(fh.read().strip().splitlines()[-1])
    return out


def scaling_table(d):
    t = ("| GPUs | c3 env-steps/s (weak: 16.7 M envs per GPU) | µs/step | per-GPU fraction of the 25 B roofline | SM clock | "
         "strong scaling (16.7 M envs in total) | e2e through host buffers (5 B/env down; 1 B/env) | c5 BFS on chip (K6), successors/s | "
         "c5 BFS hash-partitioned |\n|---|---|---|---|---|---|---|---|---|\n")
    for n, x in sorted(d.items()):
        pr, c5, ss = x["roofline"]["per_rank_frac"], x["configs"]["c5"], x.get("strong_scaling")
        frac = f"{min(pr):.3f}" if len(pr) == 1 else f"{min(pr):.3f}–{max(pr):.3f}"
        t += (f"| {n} | {f(x['value'])} | {x['ms_per_step'] * 1e3:.1f} | {frac} | {x['clocks']['sm_mhz']} MHz | "
              + (f"{f(ss['value'])} ({ss['ms_per_step'] * 1e3:.1f} µs/step, {ss['roofline_frac']:.2f})" if ss else "= weak")
              + f" | {f(x['e2e']['value'])}; {f(x['e2e']['compact_variant']['value'])} | "
              + (f"{f(c5['per_puzzle_on_chip']['value'])} ({c5['puzzles']:,} puzzles in {c5['per_puzzle_on_chip']['seconds'] * 1e3:.1f} ms)"
                 if "per_puzzle_on_chip" in c5 else "—")
              + f" | {f(c5['hash_partitioned']['value'])} ({c5['hash_partitioned']['seconds'] * 1e3:.0f} ms, "
                f"{c5['hash_partitioned']['exchange'].split(' ')[0].replace('none', 'one rank')}) |\n")
    return t


def config_table(d):
    x = d[1]
    t = (f"| Config (1×B200) | env-steps/s | µs/step | fraction of the algorithmic HBM roofline ({x['roofline']['peak']:.0f} GB/s) | "
         "bytes moved / algorithmic per env-step | steady-state DRAM traffic per launch (ncu) | parity (env-steps vs the C oracle, mismatches) |\n"
         "|---|---|---|---|---|---|---|\n")
    rows = [("c3: 6×6, 4 coloured tiles, 8 walls, 16,777,216 envs (headline)", x, x["parity"])]
    for k, label in (("c2", "c2: 5×5, 1 tile, 5 walls, 1,048,576 envs (L2-resident: 15.7 MB working set)"),
                     ("c4", "c4: 12×12, 8 coloured tiles, 36 walls, 4,194,304 envs")):
        rows.append((label, x["configs"][k], x["configs"][k]["parity"]))
    for label, r, par in rows:
        rf = r["roofline"]
        t += (f"| {label} | {f(r['value'])} | {r['ms_per_step'] * 1e3:.2f} | {rf['frac']:.3f} | "
              f"{rf['bytes_moved_per_env_step']['total']} / {rf['algorithmic_bytes_per_launch'] / r['config']['envs_per_gpu']:.0f} B | "
              + (f"{rf['traffic'] / 1e6:.1f} MB" if rf.get("traffic") else "—")
              + f" | {par['env_steps_checked']:,}: {par['mismatches'] + par['fast_path_mismatches'] + par['observation_or_valid_mask_mismatches']} |\n")
    cb = x["cpu_baseline"]
    t += (f"| reference-style Python step loop (`oracle/py_port.py`), 1 host core | {f(cb['value'])} | — | — | — | — | — |\n"
          f"| C oracle (`oracle/ts_oracle.c`), 1 host core | {f(cb['c_oracle_env_steps_per_s_1core'])} | — | — | — | — | — |\n")
    return t


def inject(path, name, text):
    with open(path) as fh:
        s = fh.read()
    pat = re.compile(rf"(<!-- BEGIN {name} -->\n).*?(<!-- END {name} -->)", re.S)
    assert pat.search(s), (path, name)
    s = pat.sub(lambda m: m.group(1) + text + m.group(2), s)
    with open(path, "w") as fh:
        fh.write(s)


def main():
    d = load()
    for doc in ("README.md", "DESIGN.md"):
        inject(os.path.join(ROOT, doc), "SCALING", scaling_table(d))
    inject(os.path.join(ROOT, "README.md"), "CONFIGS", config_table(d))
    print(scaling_table(d))
    print(config_table(d))


if __name__ == "__main__":
    main()
