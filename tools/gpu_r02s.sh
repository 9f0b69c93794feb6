#!/bin/bash
# part 1 of the evidence: suite + bench lines + launch list (small files)
T=${1:-r02s}
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/pytest_gpu_$T.log 2>&1; echo "pytest exit $?" >> gpurun_out/pytest_gpu_$T.log
python bench.py --steps 10 --warmup 3 > gpurun_out/bench_$T.json 2> gpurun_out/bench_$T.err
for c in cfg1 cfg2 cfg4 receiver; do python bench.py --config $c --steps 5 --warmup 3 > gpurun_out/bench_${T}_$c.json 2> gpurun_out/bench_${T}_$c.err; done
ncu --metrics gpu__time_duration.sum --clock-control none -s 40 -c 60 --csv --log-file gpurun_out/launches_$T.csv python bench.py --steps 2 --warmup 1 > gpurun_out/bench_under_ncu_$T.log 2>&1
tail -3 gpurun_out/pytest_gpu_$T.log
for f in bench_$T bench_${T}_cfg1 bench_${T}_cfg2 bench_${T}_cfg4 bench_${T}_receiver; do python - <<PY
import json
try:
    d=json.load(open('gpurun_out/$f.json'))
    print('$f', round(d['ms_per_step'],3), 'ms', round(d['value']), 'Msps e2e', round(d['e2e']['value']), 'roof', d['roofline']['bound'], round(d['roofline']['frac'],3), {k:round(v['avg_launch_ms'],3) for k,v in d.get('kernels',{}).items()})
except Exception as e:
    print('$f', 'FAILED', e); print(open('gpurun_out/$f.err').read()[-800:])
PY
done
