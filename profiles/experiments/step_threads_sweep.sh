# Needs commit 71e789f (the TS_STEP_THREADS / TS_STEP_MINBLOCKS switches and the variant build were removed afterwards; results: profiles/r2_step_threads_sweep.txt).
for v in "" variants/libts_thr128.so variants/libts_thr512.so "" ; do
  TS_LIB_PATH=$v python bench.py --steps 20 --warmup 5 --no-extra --no-cpu --e2e-steps 0 | python -c "import json,sys; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('$v', d['ms_per_step']*1e3, d['roofline']['frac'], d['clocks']['sm_mhz'])"
done
