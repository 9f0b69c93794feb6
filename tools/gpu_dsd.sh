#!/bin/bash
mkdir -p gpurun_out
python -m pytest tests/test_gpu_dsd_parity.py tests/test_golden.py tests/test_gpu_round2.py tests/test_gpu_host_harness.py tests/test_gpu_liquid_shim.py -m gpu -x -q 2>&1 | tail -4
python tools/probe_dsd.py | tail -1
ncu --metrics gpu__time_duration.sum --clock-control none -s 20 -c 40 --csv --log-file gpurun_out/launches_dsd_r02b.csv python tools/probe_dsd.py | tail -1
