# Needs commit 71e789f (the TS_HOST_ZERO_COPY switch was removed afterwards; results: profiles/r2_zero_copy_e2e.txt).
"""ts_step_host with the step's outputs written by the kernel straight into pinned host memory
(TS_HOST_ZERO_COPY=1) against the default (HBM + device-to-host copy per chunk):
    TS_HOST_ZERO_COPY=0 python profiles/experiments/zero_copy_e2e.py; TS_HOST_ZERO_COPY=1 python profiles/experiments/zero_copy_e2e.py"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import tiler_slider_b200 as ts  # noqa: E402

n = 16_777_216
z = os.environ.get("TS_HOST_ZERO_COPY", "0")
env = ts.BatchedTilerSliderEnv.synthetic(n, 6, 4, 8, True, seed=1002, max_steps=100, auto_reset=True)
ref = ts.BatchedTilerSliderEnv.synthetic(n, 6, 4, 8, True, seed=1002, max_steps=100, auto_reset=True)
h_act = torch.randint(0, 4, (n,), dtype=torch.uint8).pin_memory()
h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
h_flags = torch.empty(n, dtype=torch.uint8).pin_memory()
env.step_host(h_act, h_rew, h_done)
_, r, d = ref.step(h_act.cuda())
assert torch.equal(r.cpu(), h_rew) and torch.equal(d.cpu(), h_done.bool()) and torch.equal(env.pos, ref.pos), "results differ"
for name, fn in (("reward+done", lambda: env.step_host(h_act, h_rew, h_done)), ("flags only", lambda: env.step_host(h_act, h_flags=h_flags))):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        fn()
    dt = (time.perf_counter() - t0) / 20
    print(f"zero_copy={z} {name:12s} {dt * 1e3:.3f} ms/step  {n / dt:.3e} env-steps/s")
