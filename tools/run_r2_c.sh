#!/bin/bash
# round 2, GPU call C (2 GPUs): dist test with the full traceback; wide CE bring-up on GPU 0
mkdir -p gpurun_out
python -m pytest tests/test_dist_gpu.py -m gpu -x -q 2>&1 | grep -v "UserWarning\|run_backward" > gpurun_out/r2c_dist_pytest.log
grep -n "rank [01]" -A 30 gpurun_out/r2c_dist_pytest.log | cut -c1-1200 | head -60
tail -3 gpurun_out/r2c_dist_pytest.log
timeout 300 python tools/dbg_ce_wide.py check > gpurun_out/r2c_ce_check.log 2>&1
tail -20 gpurun_out/r2c_ce_check.log
timeout 300 python tools/dbg_ce_wide.py time > gpurun_out/r2c_ce_time.log 2>&1
tail -20 gpurun_out/r2c_ce_time.log
