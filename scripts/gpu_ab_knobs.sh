#!/bin/bash
mkdir -p gpurun_out
timeout 1500 python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu_fd7.log 2>&1
echo "pytest exit $?" | tee -a gpurun_out/pytest_gpu_fd7.log
tail -3 gpurun_out/pytest_gpu_fd7.log
run() { # name, env...
  name=$1; shift
  env "$@" timeout 600 python bench.py --steps 5 --warmup 3 --no-e2e --no-cpu > gpurun_out/fd7_c4_$name.json 2> gpurun_out/fd7_c4_$name.err
  python -c "import json; d=json.load(open('gpurun_out/fd7_c4_$name.json')); print('$name', d['value'], d['ms_per_step'], d['loss']['final'], d['roofline']['kernel_ms'], d['clocks']['sm_mhz'])"
}
run default CMF_X=0
run cols8 CMF_FD_COLS=8
run cols32 CMF_FD_COLS=32
run default2 CMF_X=0
timeout 600 python bench.py --config c3 --steps 10 --warmup 3 --no-e2e --no-cpu > gpurun_out/fd7_c3.json 2> gpurun_out/fd7_c3.err
python -c "import json; d=json.load(open('gpurun_out/fd7_c3.json')); print('c3', d['value'], d['ms_per_step'], d['loss'], d['roofline']['kernel_ms'])"
timeout 300 python scripts/hals_scale.py --N 512 --T 4194304 --K 128 --L 32 --iters 2 > gpurun_out/fd7_hals_c5_T4M.log 2>&1; tail -3 gpurun_out/fd7_hals_c5_T4M.log
timeout 300 python scripts/hals_scale.py --N 512 --T 1048576 --K 64 --L 32 --iters 2 > gpurun_out/fd7_hals_K64_T1M.log 2>&1; tail -3 gpurun_out/fd7_hals_K64_T1M.log
